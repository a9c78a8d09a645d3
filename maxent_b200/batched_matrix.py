"""Batched matrix-valued continuation: B independent matrices G[B, M, M, n_tau] (k-points, bootstrap samples of a
multi-orbital or Nambu Green function) continued element by element in two launches of the fused sweep in all.

``BatchedElementwiseMaxEnt`` is ``ElementwiseMaxEnt`` (python/elementwise_maxent.py) for a batch, and
``BatchedPoormanMaxEnt`` is ``PoormanMaxEnt`` (:562-653) for a batch.  Like the drop-in classes they compose two workers,
here two ``BatchedTauMaxEnt``: 'normal' entropy for the diagonal, 'plusminus' for the off-diagonal elements.  The schedule
is the one of SURVEY.md 8(e):

1. pass 1: every diagonal element (b, i, i) of every matrix in ONE ``run_device``;
2. Poorman only: ``mx_poorman_models`` builds the default model D_ij = (sqrt(A_ii A_jj) + c) delta of every needed
   off-diagonal element, and its initial vector, from pass 1's analyzer output on the device;
3. pass 2: every needed off-diagonal element (b, i, j[, re/im]) in ONE ``run_device`` (one default model per spectrum
   for Poorman).  With ``use_hermiticity`` only i < j is continued.

Every spectrum is continued by its own CTA and the default models are summed in a fixed order, so a matrix's results do
not depend on which other matrices share the batch."""
import numpy as np

from . import _lib
from .batched import ANALYZER_NAMES, BatchedTauMaxEnt

N_AN = _lib.N_ANALYZERS


def element_plan(B, M, use_hermiticity=True, use_complex=False):
    """Spectra of the two passes as int arrays of rows (b, i, j, c), c = 0 real / 1 imaginary part: the diagonal rows
    [B * M, 4] (b-major) and the off-diagonal rows [P, 4] in the order of ElementwiseMaxEnt._offdiagonal_elements
    within every matrix."""
    diag = np.array([(b, i, i, 0) for b in range(B) for i in range(M)], dtype=np.int64).reshape(-1, 4)
    parts = (0, 1) if use_complex else (0,)
    off = np.array([(b, i, j, c) for b in range(B) for i in range(M) for j in range(M)
                    if i != j and not (use_hermiticity and i > j) for c in parts], dtype=np.int64).reshape(-1, 4)
    return diag, off


def synthetic_matrix_batch(n_tau, n_omega, B, seed=7, beta=40.0, sigma=1.e-4):
    """Synthetic complex Hermitian 2x2 G(tau) batch (SURVEY.md 8(d), scaled C2): A(omega) = U diag(A_1, A_2) U^dagger
    with the Gaussian A_1 of the benchmark (C5 recipe), a second Gaussian A_2 and a random rotation U per matrix, pushed
    through the TauKernel, plus Hermitian noise of size sigma.  Returns (tau, omega, G[B, 2, 2, n_tau] complex)."""
    from .batched import synthetic_bootstrap_batch
    from .omega_meshes import HyperbolicOmegaMesh
    tau = np.linspace(0, beta, n_tau)
    omega = HyperbolicOmegaMesh(-10, 10, n_omega)
    w = np.asarray(omega)
    G1 = synthetic_bootstrap_batch(n_tau, n_omega, 1, sigma=0.0, beta=beta).numpy()[0]
    A2 = np.exp(-(w + 1.5) ** 2 / (2 * 0.7 ** 2))
    A2 /= np.sum(0.5 * (A2[1:] + A2[:-1]) * np.diff(w))
    ww, tt = np.meshgrid(w, tau)
    with np.errstate(over="ignore"):
        K = np.where(ww >= 0, -np.exp(-ww * tt) / (np.exp(-beta * ww) + 1.0),
                     -np.exp(np.minimum(ww, 0) * (beta - tt)) / (1.0 + np.exp(beta * np.minimum(ww, 0))))
    G2 = (K * (omega.delta * A2)[None, :]).sum(axis=1)
    rng = np.random.default_rng(seed)
    th, ph = rng.uniform(0.1, 0.7, B), rng.uniform(0, 2 * np.pi, B)
    c, s = np.cos(th), np.sin(th) * np.exp(1j * ph)
    G = np.empty((B, 2, 2, n_tau), dtype=complex)
    G[:, 0, 0] = (c ** 2)[:, None] * G1 + (np.abs(s) ** 2)[:, None] * G2
    G[:, 1, 1] = (np.abs(s) ** 2)[:, None] * G1 + (c ** 2)[:, None] * G2
    G[:, 0, 1] = (c * np.conj(s))[:, None] * (G1 - G2)
    n = rng.standard_normal((B, 4, n_tau))
    G[:, 0, 0] += sigma * n[:, 0]
    G[:, 1, 1] += sigma * n[:, 1]
    G[:, 0, 1] += sigma * (n[:, 2] + 1j * n[:, 3]) / np.sqrt(2.0)
    G[:, 1, 0] = np.conj(G[:, 0, 1])
    return tau, omega, G


class BatchedMatrixMaxEntResult(object):
    """Host-side result of a batched matrix run.  Arrays carry a leading batch axis:

    ``A_out`` [B, M, M, 5, n_omega] (complex with ``use_complex``; analyzer order = ANALYZER_NAMES),
    ``alpha_index`` [B, M, M, (2,) 5] (-1 = not available), ``chi2 / S / Q / probability / n_iter / converged``
    [B, M, M, (2,) n_alpha].  Elements that were not continued are NaN (-1, 0, False); with ``use_hermiticity`` the
    A_out of (j, i) is taken from (i, j), imaginary part negated, as MaxEntResult.get_A_out does.  ``zero_elements[b]``
    lists the elements skipped below G_threshold (A = 0), ``skipped_elements[b]`` the Poorman off-diagonals whose
    diagonal partner had no A_out for ``analyzer_offdiag_D`` (A = NaN).  The full A_alpha(omega) stays on the device and
    is copied on demand by ``A(b)``; ``result(b)`` (or ``out[b]``) is the MaxEntResult of matrix b."""

    def __len__(self):
        return int(self.chi2.shape[0])

    def __getitem__(self, b):
        if not -len(self) <= b < len(self):
            raise IndexError(b)
        return self.result(b % len(self))

    def _rows_of(self, b):
        """(pass, row index, (i, j, c)) of every continued element of matrix b."""
        out = []
        for k, plan in enumerate(self._plans):
            for r in np.nonzero(plan[:, 0] == b)[0]:
                out.append((k, int(r), tuple(int(x) for x in plan[r, 1:])))
        return out

    def A(self, b):
        """A_alpha(omega) of matrix b, [M, M, (2,) n_alpha, n_omega], as MaxEntResult.A assembles it: elements that were
        not continued are NaN; with ``use_hermiticity`` an element that is NaN as a whole is taken from the transposed
        one, imaginary part negated."""
        shape = self._shape + (len(self.alpha), len(self.omega))
        A = np.full(shape, np.nan)
        for k, r, (i, j, c) in self._rows_of(b):
            res = self._device[k]
            if res is not None and not self._not_run[k][r]:
                A[self._key(i, j, c)] = res.A[r].cpu().numpy()
        if self.use_hermiticity:
            M = self.matrix_structure[0]
            for i in range(M):
                for j in range(M):
                    if i != j and np.all(np.isnan(A[i, j])):
                        A[i, j] = A[j, i]
                        if self.complex_elements:
                            A[i, j, 1] = -A[i, j, 1]
        return A

    def _key(self, i, j, c):
        return (i, j, c) if self.complex_elements else (i, j)

    def result(self, b):
        """MaxEntResult of matrix b with the fields, analyzer_results[i][j][c] and zero_elements that
        PoormanMaxEnt.run() / ElementwiseMaxEnt.run() return for it."""
        from .analyzers import LineFitAnalyzer, Chi2CurvatureAnalyzer, EntropyAnalyzer, BryanAnalyzer, ClassicAnalyzer
        from .maxent_result import MaxEntResult
        out = MaxEntResult(matrix_structure=self.matrix_structure, element_wise=True, use_hermiticity=self.use_hermiticity,
                           complex_elements=self.complex_elements)
        analyzers = [LineFitAnalyzer(), Chi2CurvatureAnalyzer(), EntropyAnalyzer()]
        if self.probability_on:
            analyzers += [BryanAnalyzer(), ClassicAnalyzer()]
        out._default_analyzer_name = analyzers[0].name
        out._zero_elements = list(self.zero_elements[b])
        out.skipped_elements = list(self.skipped_elements[b])
        for k, r, (i, j, c) in self._rows_of(b):
            res = self._device[k]
            if res is None or self._not_run[k][r]:
                continue
            worker = self._workers[k]
            prob = res.problem(r)
            A = res.A[r]
            Kd = worker._K_dev * prob.delta[None, :]
            v = None if res.v is None else prob.v_to_reference_basis(res.v[r][..., :prob.n_sv]).cpu().numpy()
            key = self._key(i, j, c)
            record = dict(alpha=self.alpha, v=v, chi2=self.chi2[b][key], S=self.S[b][key], Q=self.Q[b][key],
                          A=A.cpu().numpy(), H=(A * prob.delta).cpu().numpy(), probability=self.probability[b][key],
                          omega=self.omega, G=self._G_rows[k][r], G_orig=self._G_rows[k][r], data_variable=self.tau,
                          G_rec=(A @ Kd.transpose(0, 1)).cpu().numpy(), n_iter=self.n_iter[b][key],
                          converged=self.converged[b][key], n_sv=prob.n_sv)
            out.add_sweep(record, matrix_element=(i, j), complex_index=c)
            out.analyze(analyzers, matrix_element=(i, j), complex_index=c)
        return out


class BatchedElementwiseMaxEnt(object):
    """ElementwiseMaxEnt (python/elementwise_maxent.py) for a batch of matrices G[B, M, M, n_tau] sharing tau grid,
    omega mesh, alpha mesh and kernel: the off-diagonal elements use the off-diagonal worker's own default model."""

    def __init__(self, use_hermiticity=True, use_complex=False, probability=None, reduce_singular_space=1.e-14,
                 scale_alpha="Ndata", G_threshold=1.e-10, device=None, minimizer=None):
        kw = dict(probability=probability, reduce_singular_space=reduce_singular_space, scale_alpha=scale_alpha,
                  G_threshold=G_threshold, device=device, minimizer=minimizer)
        self.maxent_diagonal = BatchedTauMaxEnt(cost_function="normal", **kw)
        self.maxent_offdiagonal = BatchedTauMaxEnt(cost_function="plusminus", **kw)
        self.use_hermiticity = bool(use_hermiticity)
        self.use_complex = bool(use_complex)
        self.probability = probability
        self.G = None
        self.tau = None
        self.error = None
        self.error_dimension = 1

    def _workers(self):
        return (self.maxent_diagonal, self.maxent_offdiagonal)

    @property
    def omega(self):
        return self.maxent_diagonal.omega

    @omega.setter
    def omega(self, value):
        for w in self._workers():
            w.omega = value

    @property
    def alpha_mesh(self):
        return self.maxent_diagonal.alpha_mesh

    @alpha_mesh.setter
    def alpha_mesh(self, value):
        for w in self._workers():
            w.alpha_mesh = value

    # ---- inputs -----------------------------------------------------------------------------------
    def set_G_tau_data(self, tau, G):
        """tau[n_tau], G[B, M, M, n_tau] (numpy or torch; complex allowed, its imaginary part is used with
        ``use_complex`` only, as in ElementwiseMaxEnt.set_G_tau_data)."""
        if G.ndim != 4 or G.shape[1] != G.shape[2]:
            raise ValueError("G must be [B, M, M, n_tau], got shape %s" % (tuple(G.shape),))
        if G.shape[-1] != len(tau):
            raise Exception("tau and G_tau don't have the same length")
        for w in self._workers():
            w.set_G_tau_data(tau, np.zeros((1, len(tau))))
            w.G = None
        self.tau = np.asarray(tau, dtype=np.float64)
        self.G = G

    def set_error(self, error, per_spectrum=None):
        """A scalar or a vector [n_tau] for every element; an array [M, M, n_tau] with one error vector per element
        (one whitening group per element); an array [B, M, M] with one scalar error bar per spectrum.  An array that
        fits both 3-D shapes is read as per element unless ``per_spectrum=True``."""
        self.error, self.error_dimension, self._per_spectrum = error, 1, per_spectrum

    def set_cov(self, cov):
        """Covariance [n_tau, n_tau] shared by every element.  Per-element covariances are not supported."""
        cov = np.asarray(cov, dtype=np.float64)
        if cov.ndim != 2:
            raise NotImplementedError("per-element covariance matrices [M, N, n_tau, n_tau] are not supported by the "
                                      "batched matrix path; use PoormanMaxEnt / ElementwiseMaxEnt per matrix")
        self.error, self.error_dimension = cov, 2

    def _error_kind(self, B, M):
        """'shared' | 'element' | 'spectrum' | 'cov' for the error set by set_error / set_cov (validates the shape)."""
        if self.error is None:
            raise Exception("no error set: call set_error or set_cov")
        if self.error_dimension == 2:
            return "cov"
        n_tau = len(self.tau)
        e = np.asarray(self.error, dtype=np.float64)
        if e.ndim == 0 or e.shape == (n_tau,):
            return "shared"
        if e.shape == (M, M, n_tau) and not self._per_spectrum:
            return "element"
        if e.shape == (B, M, M):
            return "spectrum"
        raise ValueError("error of shape %s: expected a scalar, [n_tau] = [%d], [M, M, n_tau] = %s or [B, M, M] = %s"
                         % (e.shape, n_tau, (M, M, n_tau), (B, M, M)))

    def _put_error(self, worker, kind, plan):
        """Error model of the spectra `plan` (rows (b, i, j, c)) on `worker` (unchanged inputs keep the worker's
        prepared problems)."""
        key = (kind, plan.tobytes())
        last = getattr(worker, "_matrix_error", None)
        if last is not None and last[0] is self.error and last[1] == key:
            return
        worker._matrix_error = (self.error, key)
        if kind == "cov":
            worker.set_cov(self.error)
            return
        e = np.asarray(self.error, dtype=np.float64)
        if kind == "shared":
            worker.set_error(e, per_spectrum=False)
        elif kind == "spectrum":
            worker.set_error(e[plan[:, 0], plan[:, 1], plan[:, 2]], per_spectrum=True)
        else:                                             # whitening group = matrix element
            elems, index = np.unique(plan[:, 1:3], axis=0, return_inverse=True)
            worker.set_error_groups(e[elems[:, 0], elems[:, 1]], np.asarray(index).reshape(-1))

    # ---- run --------------------------------------------------------------------------------------
    def _G_device(self):
        import torch
        dev = self.maxent_diagonal.prepare().device
        G = self.G if torch.is_tensor(self.G) else torch.from_numpy(np.ascontiguousarray(self.G))
        G = G.to(dev, non_blocking=True)
        if not G.is_complex():
            G = G.to(torch.float64)
            return torch.stack([G, torch.zeros_like(G)], dim=-1)
        return torch.view_as_real(G.to(torch.complex128))

    @staticmethod
    def _gather(Gri, plan):
        """Rows G[b, i, j, :, c] of the planned spectra, gathered on the device: [P, n_tau]."""
        import torch
        idx = [torch.as_tensor(plan[:, k], device=Gri.device) for k in range(4)]
        return Gri[idx[0], idx[1], idx[2], :, idx[3]].contiguous()

    def set_preblur(self, *args, **kwargs):
        raise NotImplementedError("preblur is not supported by the batched matrix path; use ElementwiseMaxEnt per matrix")

    def _check(self):
        if self.G is None:
            raise Exception("no data: call set_G_tau_data")

    def _offdiagonal_models(self, diag_res, off_plan, G2):
        """Default models of the off-diagonal pass: (G2, D, v0, not_ok) -- the worker's own model here."""
        return G2, None, None, None

    def run_diagonal(self):
        """Pass 1 only (DiagonalMaxEnt): every diagonal element of every matrix."""
        return self._run(diagonal_only=True)

    def run(self):
        return self._run(diagonal_only=False)

    def run_device(self, timeline=None, diagonal_only=False):
        """The two passes on the device: (plans, (pass-1 SweepResult, pass-2 SweepResult or None), G rows, not_ok).
        ``timeline`` (a list) receives CUDA events recorded before pass 1, after pass 1, after the gather of the pass-2
        rows, after the default models and after pass 2 (tools/matrix_bench.py)."""
        import torch
        self._check()
        B, M = int(self.G.shape[0]), int(self.G.shape[1])
        kind = self._error_kind(B, M)
        diag_plan, off_plan = element_plan(B, M, self.use_hermiticity, self.use_complex)
        if diagonal_only:
            off_plan = off_plan[:0]
        self._put_error(self.maxent_diagonal, kind, diag_plan)
        if len(off_plan):
            self._put_error(self.maxent_offdiagonal, kind, off_plan)
        dev = self.maxent_diagonal.prepare().device

        def mark():
            if timeline is not None:
                ev = torch.cuda.Event(enable_timing=True)
                ev.record(torch.cuda.current_stream(dev))
                timeline.append(ev)
        with torch.cuda.device(dev):
            Gri = self._G_device()
            G1 = self._gather(Gri, diag_plan)
            mark()
            r1 = self.maxent_diagonal.run_device(G1, want_A=True, want_v=True, skip_small=True)
            mark()
            if len(off_plan) == 0:
                return (diag_plan, off_plan), (r1, None), (G1, None), None
            G2 = self._gather(Gri, off_plan)
            mark()
            G2, D, v0, not_ok = self._offdiagonal_models(r1, off_plan, G2)
            mark()
            r2 = self.maxent_offdiagonal.run_device(G2, want_A=True, want_v=True, D=D, v0=v0, skip_small=True)
            mark()
        return (diag_plan, off_plan), (r1, r2), (G1, G2), not_ok

    def _run(self, diagonal_only):
        import torch
        plans, results, G_rows, not_ok = self.run_device(diagonal_only=diagonal_only)
        B, M = int(self.G.shape[0]), int(self.G.shape[1])
        out = BatchedMatrixMaxEntResult()
        out.matrix_structure = (M, M)
        out.use_hermiticity, out.complex_elements = self.use_hermiticity, self.use_complex
        out.probability_on = self.probability is not None
        out.omega, out.tau = self.omega, self.tau
        out.alpha = self.maxent_diagonal.alpha_effective()
        out._plans, out._device = plans, results
        out._workers = self._workers()
        out._shape = (M, M) + ((2,) if self.use_complex else ())
        not_run, host = [], []
        for k, (plan, res) in enumerate(zip(plans, results)):
            if res is None:
                not_run.append(np.zeros(0, dtype=bool))
                host.append(None)
                continue
            got = {name: getattr(res, name).cpu().numpy() for name in
                   ("chi2", "S", "Q", "logp", "n_iter", "status", "alpha_index", "A_out")}
            skipped = (got["status"][:, 0] & _lib.STATUS_SKIPPED) != 0
            bad = np.zeros(len(plan), dtype=bool) if (k == 0 or not_ok is None) else ~not_ok.cpu().numpy().astype(bool)
            got["zero"], got["bad"] = skipped & ~bad, bad
            not_run.append(skipped)
            host.append(got)
        out._not_run = not_run
        out._G_rows = [None if g is None else g.cpu().numpy() for g in G_rows]
        self._fill(out, plans, host, B, M)
        return out

    def _fill(self, out, plans, host, B, M):
        n_alpha, n_omega = len(out.alpha), len(self.omega)
        shp = (B,) + out._shape
        out.chi2, out.S, out.Q, out.probability = (np.full(shp + (n_alpha,), np.nan) for _ in range(4))
        out.n_iter = np.zeros(shp + (n_alpha,), dtype=np.int32)
        out.converged = np.zeros(shp + (n_alpha,), dtype=bool)
        out.alpha_index = np.full(shp + (N_AN,), -1, dtype=np.int32)
        A_out = np.full(shp + (N_AN, n_omega), np.nan)
        computed = np.zeros(shp, dtype=bool)
        out.zero_elements = [[] for _ in range(B)]
        out.skipped_elements = [[] for _ in range(B)]
        zeros = []
        for k, (plan, got) in enumerate(zip(plans, host)):
            if got is None:
                continue
            for r, row in enumerate(plan):
                b, i, j, c = (int(x) for x in row)
                key = (b, i, j, c) if self.use_complex else (b, i, j)
                if got["bad"][r]:
                    out.skipped_elements[b].append((i, j) + ((c,) if self.use_complex else ()))
                    continue
                if got["zero"][r]:
                    if (i, j) not in out.zero_elements[b]:
                        out.zero_elements[b].append((i, j))       # MaxEntLoop.run_jobs lists the element, not the part
                    zeros.append((b, i, j))
                    continue
                out.chi2[key], out.S[key], out.Q[key] = got["chi2"][r], got["S"][r], got["Q"][r]
                out.probability[key] = got["logp"][r]
                out.n_iter[key] = got["n_iter"][r]
                out.converged[key] = (got["status"][r] & _lib.STATUS_CONVERGED) != 0
                out.alpha_index[key] = got["alpha_index"][r]
                A_out[key] = got["A_out"][r]
                computed[key] = True
            if k == 0 and self.use_complex:                      # a Hermitian matrix has a real diagonal
                for b in range(B):
                    for i in range(M):
                        out.zero_elements[b].append((i, i, 1))
                        zeros.append((b, i, i, 1))
        # MaxEntResult.get_A_out: zero for the listed elements, then every computed part, then (use_hermiticity) every
        # part that was not computed is taken from the computed transposed part, imaginary part negated
        for key in zeros:
            A_out[key] = np.where(np.asarray(computed[key])[..., None, None], A_out[key], 0.0)
        if self.use_hermiticity:
            A4, C4 = (A_out, computed) if self.use_complex else (A_out[:, :, :, None], computed[..., None])
            for b, i, j, c in zip(*np.nonzero(~C4)):
                if i != j and C4[b, j, i, c]:
                    A4[b, i, j, c] = (-1.0 if self.use_complex and c == 1 else 1.0) * A4[b, j, i, c]
        out.A_out = A_out[..., 0, :, :] + 1j * A_out[..., 1, :, :] if self.use_complex else A_out


class BatchedPoormanMaxEnt(BatchedElementwiseMaxEnt):
    """PoormanMaxEnt (python/elementwise_maxent.py:562-653) for a batch: the off-diagonal element (i, j) of matrix b uses
    the default model (sqrt(A_ii A_jj) + D_add_constant) delta built on the device from the diagonal results of
    ``analyzer_offdiag_D`` (mx_poorman_models).  An off-diagonal element whose diagonal partner has no A_out for that
    analyzer is not continued (NaN, ``skipped_elements``)."""

    def __init__(self, use_hermiticity=True, use_complex=False, analyzer_offdiag_D="LineFitAnalyzer", D_add_constant=1.e-6,
                 reduce_singular_space=1.e-14, probability=None, minimizer=None, **kwargs):
        super(BatchedPoormanMaxEnt, self).__init__(use_hermiticity=use_hermiticity, use_complex=use_complex,
                                                   probability=probability, reduce_singular_space=reduce_singular_space,
                                                   minimizer=minimizer, **kwargs)
        if analyzer_offdiag_D not in ANALYZER_NAMES:
            raise ValueError("analyzer_offdiag_D must be one of %s" % (ANALYZER_NAMES,))
        self.analyzer_offdiag_D = analyzer_offdiag_D
        self.D_add_constant = D_add_constant

    def default_models(self, A_out, off_plan):
        """mx_poorman_models on pass-1 output: A_out [B * M, 5, n_omega] (device, rows in the order of the diagonal plan)
        and the off-diagonal plan [P, 4] (b, i, j, c) -> (D [P, ldD], v0 [P, n_sv], ok [P]) on the device."""
        import torch
        off = self.maxent_offdiagonal
        M = int(self.G.shape[1])
        self._put_error(off, self._error_kind(int(self.G.shape[0]), M), off_plan)
        prob = off.prepare()
        dev = prob.device
        P = int(off_plan.shape[0])
        # indices the kernel dereferences stay on the host: the operator checks them there before the upload
        rows = torch.from_numpy(np.stack([off_plan[:, 0] * M + off_plan[:, 1], off_plan[:, 0] * M + off_plan[:, 2]],
                                         axis=1).astype(np.int32))
        plan = off._batch_plan(P)
        Vp = torch.stack([q.Vp for q in plan.problems]).contiguous()
        group = None if plan.index is None else torch.from_numpy(np.asarray(plan.index).astype(np.int32))
        A_init = None if off.A_init is None else torch.as_tensor(np.asarray(off.A_init, dtype=np.float64), device=dev)
        ld = (prob.n_omega + 1) & ~1
        D = torch.empty((P, ld), dtype=torch.float64, device=dev)
        v0 = torch.empty((P, int(Vp.shape[2])), dtype=torch.float64, device=dev)
        ok = torch.empty((P,), dtype=torch.int32, device=dev)
        from . import ops
        ops.poorman_models(A_out, ANALYZER_NAMES.index(self.analyzer_offdiag_D), rows, prob.delta,
                           float(self.D_add_constant), A_init, Vp, group, D, v0, ok)
        return D, v0, ok

    def _offdiagonal_models(self, diag_res, off_plan, G2):
        import torch
        # a diagonal element below G_threshold has no analyzer output: NaN rows make its partners ok = 0
        skipped = (diag_res.status[:, 0] & _lib.STATUS_SKIPPED) != 0
        diag_res.A_out.masked_fill_(skipped[:, None, None], float("nan"))
        D, v0, ok = self.default_models(diag_res.A_out, off_plan)
        # an element without a default model is left out of the launch by the threshold skip of run_device
        G2 = torch.where(ok[:, None] != 0, G2, torch.zeros_like(G2))
        return G2, D, v0, ok
