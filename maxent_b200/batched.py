"""Batched front end: many independent spectra that share one kernel (k-points, orbital elements,
bootstrap samples) continued in ONE fused launch per GPU.

The reference has no counterpart: "many spectra" is a Python ``for`` loop over ``TauMaxEnt.run``
(doc/guide/blockgf.rst:10-18, python/elementwise_maxent.py:236-268).  This class sits beside the
drop-in single-spectrum API and uses the same vocabulary (``set_G_tau_data``, ``set_error``, ``omega``,
``alpha_mesh``, ``D``, ``reduce_singular_space``, ``scale_alpha``, ``G_threshold``).

Multi-GPU: one process per GPU, each owning a contiguous shard of the batch (``shard_bounds``); the only
collective is the final gather of the result arrays (``gather_results``).
"""
import ctypes

import numpy as np

from . import _lib, engine
from .alpha_meshes import LogAlphaMesh
from .default_models import FlatDefaultModel
from .omega_meshes import HyperbolicOmegaMesh, DataOmegaMesh

ANALYZER_NAMES = ("LineFitAnalyzer", "Chi2CurvatureAnalyzer", "EntropyAnalyzer", "ClassicAnalyzer", "BryanAnalyzer")


def hyperbolic_omega(omega_min, omega_max, n_points):
    return HyperbolicOmegaMesh(omega_min, omega_max, n_points)


def shard_bounds(n_total, world_size, rank):
    """Contiguous, balanced split of ``n_total`` spectra over ``world_size`` ranks: [lo, hi) of ``rank``."""
    base, rem = divmod(int(n_total), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def synthetic_bootstrap_batch(n_tau, n_omega, n_spectra, first=0, seed=5, beta=40.0, mu=1.0, width=0.5,
                              sigma=1.e-4, pin=False):
    """Synthetic G(tau) batch of the benchmark (SURVEY.md 8(d) C5): a Gaussian A(omega) pushed through
    the TauKernel plus sigma * N(0,1) noise, rows [first, first + n_spectra) of the seeded noise matrix.
    Returns a (pinned) host float64 tensor [n_spectra, n_tau]."""
    import torch
    tau = np.linspace(0, beta, n_tau)
    omega = HyperbolicOmegaMesh(-10, 10, n_omega)
    w = np.asarray(omega)
    A = np.exp(-(w - mu) ** 2 / (2 * width ** 2))
    A /= np.sum(0.5 * (A[1:] + A[:-1]) * np.diff(w))
    ww, tt = np.meshgrid(w, tau)
    with np.errstate(over="ignore"):
        K = np.where(ww >= 0, -np.exp(-ww * tt) / (np.exp(-beta * ww) + 1.0),
                     -np.exp(np.minimum(ww, 0) * (beta - tt)) / (1.0 + np.exp(beta * np.minimum(ww, 0))))
    # fixed summation order: numpy's (single-threaded, pairwise) reduction instead of a BLAS GEMV whose blocking -- and
    # therefore the last bits of G -- depends on the thread count of the host (torchrun sets OMP_NUM_THREADS=1, a plain
    # run does not: round 1 saw 887.88 vs 887.80 LM iterations per spectrum for "the same" batch)
    G_exact = (K * (omega.delta * A)[None, :]).sum(axis=1)
    rng = np.random.default_rng(seed)
    if first:
        # rows [0, first) belong to lower ranks: skip them in blocks instead of materialising them
        left = first
        while left > 0:
            blk = min(left, 4096)
            rng.standard_normal((blk, n_tau))
            left -= blk
    G = G_exact[None, :] + sigma * rng.standard_normal((n_spectra, n_tau))
    t = torch.from_numpy(np.ascontiguousarray(G))
    return t.pin_memory() if pin and torch.cuda.is_available() else t


class BatchedMaxEntResult(object):
    """Host-side result of one batched run.  Arrays are numpy views of pinned host buffers:

    ``alpha`` [n_alpha] (scaled alpha actually used), ``chi2 / S / Q / probability`` [B, n_alpha],
    ``n_iter`` [B, n_alpha], ``converged`` [B, n_alpha], ``alpha_index`` [B, 5] (-1 = analyzer not available),
    ``A_out`` [B, 5, n_omega] (analyzer order = ANALYZER_NAMES), ``zero_elements`` = indices skipped because
    max|G| < G_threshold (python/maxent_loop.py:174-179).  The full A_alpha(omega) stays on the device in
    ``device.A`` [B, n_alpha, n_omega] and is copied on demand by ``A(b)``."""

    def __init__(self):
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    def A(self, b):
        return self.device.A[b].cpu().numpy()

    def __len__(self):
        return int(self.chi2.shape[0])

    def __getitem__(self, b):
        """``result[b]`` = ``result.spectrum(b)``."""
        if not -len(self) <= b < len(self):
            raise IndexError(b)
        return self.spectrum(b % len(self))

    def analyzer(self, name):
        k = ANALYZER_NAMES.index(name)
        return dict(alpha_index=self.alpha_index[:, k], A_out=self.A_out[:, k])

    def spectrum(self, b):
        """Per-spectrum dict with the field names of MaxEntResultData (python/maxent_result.py:181-188)."""
        d = dict(alpha=self.alpha, chi2=self.chi2[b], S=self.S[b], Q=self.Q[b], probability=self.probability[b],
                 A=self.A(b), omega=self.omega, n_iter=self.n_iter[b], converged=self.converged[b])
        d["analyzer_results"] = {n: dict(alpha_index=int(self.alpha_index[b, k]), A_out=self.A_out[b, k])
                                 for k, n in enumerate(ANALYZER_NAMES) if self.alpha_index[b, k] >= 0}
        return d


class _BatchPlan(object):
    """The error model of one launch: ``problems`` (its SharedProblems; the base problem alone without whitening groups),
    ``index`` [B] (host: every spectrum's problem) or None, ``sigma`` [B] or None, ``alpha`` (the mesh the sweep gets),
    ``alpha_scale`` [B] or None, and ``rotations``: per group the rotation T of the data of a covariance group, or None."""

    def __init__(self, problems, index, sigma, alpha, alpha_scale=None, rotations=None):
        self.problems, self.index, self.sigma = problems, index, sigma
        self.alpha, self.alpha_scale, self.rotations = alpha, alpha_scale, rotations

    def subset(self, rows):
        """The plan of the spectra `rows` (host indices): the same problems under the same numbering."""
        take = lambda x: None if x is None else x[rows]
        return _BatchPlan(self.problems, take(self.index), take(self.sigma), self.alpha, take(self.alpha_scale),
                          self.rotations)


class BatchedTauMaxEnt(object):
    """MaxEnt continuation of a batch G[B, n_tau] sharing tau grid, omega mesh, error model and alpha mesh.

    Matsubara data G(i omega_n)[B, n_iw] (``set_G_iw_data``) enter as the stacked real rows [Re G; Im G] of the
    IOmegaKernel (python/kernels.py:283-346, ``kernels.IOmegaKernel.fused_matrix``); A(omega) stays real.

    Parameters mirror MaxEntLoop.__init__ (python/maxent_loop.py:83-94): ``cost_function`` in
    {'normal', 'plusminus', 'bryan'}, ``probability`` in {None, 'normal'}, ``reduce_singular_space``,
    ``scale_alpha`` ('Ndata' | number | None), ``G_threshold``."""

    launches_per_step = 3          # mx_project_data, mx_alpha_sweep, mx_analyze

    def __init__(self, cost_function="normal", probability=None, reduce_singular_space=1.e-14,
                 scale_alpha="Ndata", G_threshold=1.e-10, device=None, svd="jacobi", minimizer=None):
        if cost_function not in _lib.VARIANTS:
            raise Exception("unknown cost_function %r for the batched path" % (cost_function,))
        if probability not in (None, "normal"):
            raise Exception("unknown probability %r" % (probability,))
        self.cost_function = cost_function
        self.probability = probability
        self.reduce_singular_space = reduce_singular_space
        self.scale_alpha = scale_alpha
        self.G_threshold = G_threshold
        self.device = device
        self.svd = svd
        # engine.LMParams, or a LevenbergMinimizer like the one MaxEntLoop takes (python/maxent_loop.py:83-94)
        self.minimizer = (engine.LMParams() if minimizer is None else
                          minimizer.lm_params() if hasattr(minimizer, "lm_params") else minimizer)
        self.omega = HyperbolicOmegaMesh(-10, 10, 100)
        self.alpha_mesh = LogAlphaMesh(1e-4, 20, 20)
        self.D = None
        self.A_init = None
        self.tau = None
        self.beta = None
        self.iomega = None                # Matsubara frequencies nu_n: the kernel is IOmegaKernel(iomega, omega)
        self.K = None                     # explicit kernel matrix (DataKernel) or None -> TauKernel(tau, omega, beta)
        self.err = None
        self.cov = None
        self._per_spectrum = None
        self._groups = None               # set_error_groups: the group of every spectrum
        self._group_cache = {}            # content of a whitening group -> its SharedProblem
        self.G = None
        self.problem = None
        self.gamma, self.linefit_deg, self.bryan_by_integration = 0.2, 0, False

    # ---- inputs -----------------------------------------------------------------------------------
    def set_kernel_tau(self, tau, omega=None, beta=None):
        self.tau = np.asarray(tau, dtype=np.float64)
        self.beta = float(self.tau[-1] if beta is None else beta)
        if omega is not None:
            self.omega = omega if hasattr(omega, "delta") else DataOmegaMesh(omega)
        self.K = None
        self.iomega = None
        self.problem = None

    def set_kernel_iw(self, iomega, omega=None):
        """IOmegaKernel (python/kernels.py:283-346): K(i nu_n, omega) = 1 / (i nu_n - omega), ``iomega`` = the real
        Matsubara frequencies nu_n.  The sweep sees the stacked real kernel [Re K; Im K] (2 n_iw rows)."""
        iomega = np.array(iomega, dtype=np.float64).reshape(-1)
        if len(iomega) < 1:
            raise Exception("no Matsubara frequencies")
        if self.cov is not None:
            raise NotImplementedError("a covariance matrix of Matsubara data is not supported (IOmegaKernel.transform)")
        self.iomega = iomega
        if omega is not None:
            self.omega = omega if hasattr(omega, "delta") else DataOmegaMesh(omega)
        self.tau = self.beta = self.K = None
        self.problem = None

    def set_kernel_data(self, K, omega):
        """DataKernel (python/kernels.py:183-207): K[n_tau, n_omega] verbatim."""
        self.K = np.asarray(K, dtype=np.float64)
        self.omega = omega if hasattr(omega, "delta") else DataOmegaMesh(omega)
        self.iomega = None
        self.problem = None

    def set_alpha_mesh_log(self, alpha_min, alpha_max, n_points):
        self.alpha_mesh = LogAlphaMesh(alpha_min, alpha_max, n_points)

    def set_G_tau_data(self, tau, G):
        """tau[n_tau], G[B, n_tau] (python/tau_maxent.py:181-196, batched)."""
        G = np.asarray(G) if not hasattr(G, "data_ptr") else G
        if G.is_complex() if hasattr(G, "is_complex") else np.iscomplexobj(G):
            raise NotImplementedError("complex G(tau) is not continued by BatchedTauMaxEnt: Matsubara data go through "
                                      "set_G_iw_data, complex matrix elements through BatchedElementwiseMaxEnt")
        if G.shape[-1] != len(tau):
            raise Exception("tau and G_tau don't have the same length")
        if self.tau is None or len(self.tau) != len(tau) or np.any(self.tau != np.asarray(tau)):
            self.set_kernel_tau(tau, None, None)
        self.G = G

    def set_G_iw_data(self, iomega, G_iw):
        """iomega[n_iw] (real Matsubara frequencies), G_iw[B, n_iw] complex (numpy or tensor): kept as the stacked real
        rows [Re G_iw, Im G_iw] of [B, 2 n_iw] that the IOmegaKernel's fused matrix continues."""
        iomega = np.asarray(iomega, dtype=np.float64).reshape(-1)
        if hasattr(G_iw, "data_ptr"):
            import torch
            G = G_iw if G_iw.dim() > 1 else G_iw[None, :]
            if G.dim() != 2:
                raise NotImplementedError("G_iw must be [B, n_iw]: matrix-valued Matsubara data are not supported")
            G = torch.cat([G.real, G.imag] if G.is_complex() else [G, torch.zeros_like(G)], dim=1).to(torch.float64)
        else:
            G = np.asarray(G_iw)
            G = G if G.ndim > 1 else G[None, :]
            if G.ndim != 2:
                raise NotImplementedError("G_iw must be [B, n_iw]: matrix-valued Matsubara data are not supported")
            G = np.ascontiguousarray(np.concatenate([G.real, G.imag], axis=1), dtype=np.float64)
        if G.shape[1] != 2 * len(iomega):
            raise Exception("iomega and G_iw don't have the same length")
        if self.iomega is None or len(self.iomega) != len(iomega) or np.any(self.iomega != iomega):
            self.set_kernel_iw(iomega, None)
        self.G = G

    def set_error(self, err, per_spectrum=None):
        """Error bars of the data (python/tau_maxent.py:227-251), for the batch:

        * a scalar, or a vector [n_tau] -- shared by every spectrum;
        * a vector [B] (``per_spectrum=True`` if B == n_tau) -- one scalar error bar per spectrum (bootstrap / QMC
          batches): same singular space, Xi_b = S / sigma_b, still one launch;
        * an array [B, n_tau] -- one error vector per spectrum: spectra with identical vectors form a group with its own
          whitening rotation V' = V_s P_g; all groups run in ONE launch of the sweep (MxProblem.vt_index)."""
        self.err = err
        self.cov = None
        self._per_spectrum = per_spectrum
        self._groups = None
        self.problem = None
        self._group_cache = {}

    def set_error_groups(self, err, index):
        """Whitening groups given directly: ``err`` [G, n_tau] holds G error vectors and ``index`` [B] the group of every
        spectrum -- the [B, n_tau] case of ``set_error`` without the copy per spectrum (the batched matrix front ends map
        per-element error vectors to groups by element index)."""
        self.set_error(np.asarray(err, dtype=np.float64))
        self._groups = np.asarray(index, dtype=np.int64).reshape(-1)

    def set_cov(self, cov, cov_threshold=1.e-14):
        """Covariance matrix of the data, [n_tau, n_tau] shared by the batch or [B, n_tau, n_tau] per spectrum
        (TauMaxEnt.set_cov, python/tau_maxent.py:253-288): rotate into the eigenbasis, errors = sqrt(eigenvalues),
        eigenvalues below ``cov_threshold`` dropped.  Identical matrices share one whitening group."""
        if self.iomega is not None:
            raise NotImplementedError("a covariance matrix of Matsubara data is not supported (IOmegaKernel.transform)")
        cov = np.asarray(cov, dtype=np.float64)
        assert np.max(np.abs(cov - np.swapaxes(cov, -1, -2))) < 1.e-10, 'Supplied covariance matrix is not symmetric.'
        self.cov = cov
        self.cov_threshold = cov_threshold
        self.err = None
        self._groups = None
        self.problem = None
        self._group_cache = {}

    def _error_plan(self, B):
        """The error model of B spectra, worked out on the host: ('shared', None, None) | ('sigma', sigma[B], None) |
        ('groups', index[B], specs) with one spec = (T or None, error vector) per whitening group.  The groups of
        err[B, n_tau] are numbered in the sorted order of their vectors, those of cov[B, n, n] in the order of first
        appearance."""
        n_tau = self._n_rows()
        if self.cov is not None:
            covs = self.cov if self.cov.ndim == 3 else self.cov[None]
            if self.cov.ndim == 3 and covs.shape[0] != B:
                raise Exception("%d covariance matrices for %d spectra" % (covs.shape[0], B))
            keys, specs, index = {}, [], np.zeros(B, dtype=np.int64)
            for b in range(covs.shape[0]):
                k = hash(covs[b].tobytes())
                if k not in keys:
                    e, v = np.linalg.eigh(covs[b])
                    keep = e >= self.cov_threshold
                    keys[k] = len(specs)
                    specs.append((np.ascontiguousarray(v[:, keep].conjugate().T), np.sqrt(e[keep])))
                index[b] = keys[k]
            if self.cov.ndim == 2:
                index[:] = 0
            return "groups", index, specs
        if self.err is None:
            raise Exception("no error set: call set_error")
        err, per_spectrum = self._row_error()
        if self._groups is not None:
            if self._groups.shape != (B,) or err.ndim != 2 or err.shape[1] != n_tau:
                raise Exception("error groups: %s vectors for %d spectra, index %s" % (err.shape, B, self._groups.shape))
            return "groups", self._groups, [(None, e) for e in err]
        if err.ndim == 0 or (err.ndim == 1 and err.shape[0] == n_tau and not per_spectrum):
            return "shared", None, None
        if err.ndim == 1:
            if err.shape[0] != B:
                raise Exception("Supply a scalar error, one per tau point, one per spectrum, or an array [B, n_tau].")
            return "sigma", err, None
        if err.shape != (B, n_tau):
            raise Exception("error array has shape %s, data has %s" % (err.shape, (B, n_tau)))
        uniq, index = np.unique(err, axis=0, return_inverse=True)
        return "groups", np.asarray(index).reshape(-1), [(None, u) for u in uniq]

    def _batch_plan(self, B):
        """The error model of a launch over B spectra (_error_plan) with the SharedProblem of every group and the
        alpha mesh; computed on the whole batch, so that a spectrum's group does not depend on which others are live."""
        mode, a, specs = self._error_plan(B)
        plan = _BatchPlan([self.prepare()], None, a if mode == "sigma" else None, self.alpha_effective())
        if mode != "groups":
            return plan
        plan.index = index = a
        plan.problems = [self._group_problem(spec) for spec in specs]
        if specs[0][0] is not None:
            plan.rotations = [T for T, _ in specs]
        rows = [q.n_tau for q in plan.problems]
        if isinstance(self.scale_alpha, str) and len(set(rows)) > 1:
            # scale_alpha = 'Ndata' counts the rows of the ROTATED data (python/maxent_loop.py:216-220, after set_cov):
            # groups whose covariance dropped eigenvalues get their own factor
            plan.alpha = np.asarray(self.alpha_mesh, dtype=np.float64)
            plan.alpha_scale = np.array([rows[g] for g in index], dtype=np.float64)
        elif isinstance(self.scale_alpha, str):
            plan.alpha = np.asarray(self.alpha_mesh, dtype=np.float64) * self._n_data(rows[0])
        return plan

    def _n_rows(self):
        """Rows of the data the sweep sees: n_tau, or 2 n_iw stacked rows of Matsubara data."""
        if self.iomega is not None:
            return 2 * len(self.iomega)
        return len(self.tau) if self.tau is not None else self.K.shape[0]

    def _n_data(self, n_rows):
        """The number of data points scale_alpha = 'Ndata' counts for n_rows rows: Matsubara data count their complex
        points, len(G) of MaxEntLoop._scale (python/maxent_loop.py:216-220), not the stacked rows."""
        return n_rows // 2 if self.iomega is not None else n_rows

    def _row_error(self):
        """(err, per_spectrum) in the rows the sweep sees: an error per Matsubara point ([n_iw] or [G, n_iw]) is repeated
        for the Re and Im rows (IOmegaKernel.stack); for Matsubara data a 1-D error not of length n_iw is one per
        spectrum."""
        err = np.asarray(self.err, dtype=np.float64)
        if self.iomega is None or err.ndim == 0:
            return err, self._per_spectrum
        n_iw = len(self.iomega)
        if err.ndim == 1 and (self._per_spectrum or err.shape[0] != n_iw):
            return err, True
        if err.shape[-1] != n_iw:
            raise Exception("error array has shape %s, the data have %d Matsubara points" % (err.shape, n_iw))
        return np.concatenate([err, err], axis=-1), False

    # ---- run --------------------------------------------------------------------------------------
    def prepare(self):
        """Everything that depends on the kernel only (KernelSVD, truncation, layout); cached, and rebuilt when one of the
        public attributes it depends on was replaced (D, A_init, omega, reduce_singular_space, cost_function, svd)."""
        key = (self.cost_function, None if self.reduce_singular_space is None else float(self.reduce_singular_space), self.svd,
               id(self.omega), id(self.D), id(self.A_init), id(self.K), id(self.tau), self.beta, id(self.iomega))
        if self.problem is not None and getattr(self, "_problem_key", None) == key:
            return self.problem
        self._problem_key = key
        self._group_cache = {}
        import torch
        if not torch.cuda.is_available():
            raise _lib.MaxEntLibraryError("maxent_b200 needs a CUDA device (no CPU fallback)")
        dev = torch.device("cuda" if self.device is None else self.device)
        lib = _lib.load()
        omega = self.omega
        with torch.cuda.device(dev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            if self.iomega is not None:
                i_d = torch.as_tensor(self.iomega, device=dev)
                o_d = torch.as_tensor(np.asarray(omega, dtype=np.float64), device=dev)
                K = torch.empty((2 * len(self.iomega), len(omega)), dtype=torch.float64, device=dev)
                _lib.check(lib.mx_iomega_kernel(i_d.data_ptr(), o_d.data_ptr(), len(self.iomega), len(omega),
                                                K.data_ptr(), stream), "mx_iomega_kernel")
            elif self.K is None:
                if self.tau is None:
                    raise Exception("no kernel: call set_G_tau_data / set_G_iw_data / set_kernel_tau / set_kernel_data "
                                    "first")
                t_d = torch.as_tensor(self.tau, device=dev)
                o_d = torch.as_tensor(np.asarray(omega, dtype=np.float64), device=dev)
                K = torch.empty((len(self.tau), len(omega)), dtype=torch.float64, device=dev)
                _lib.check(lib.mx_tau_kernel(t_d.data_ptr(), o_d.data_ptr(), len(self.tau), len(omega), self.beta,
                                             K.data_ptr(), stream), "mx_tau_kernel")
            else:
                K = torch.as_tensor(self.K, device=dev)
        if self.err is None and self.cov is None:
            raise Exception("no error set: call set_error")
        D = FlatDefaultModel(omega).D if self.D is None else (self.D.D if hasattr(self.D, "D") else np.asarray(self.D))
        err, per_spectrum = self._row_error() if self.err is not None else (np.float64(1.0), None)
        shared = err.ndim == 0 or (err.ndim == 1 and err.shape[0] == K.shape[0] and not per_spectrum)
        # per-spectrum error models: the base problem carries err = 1 (kernel SVD, truncation, V layout); error scales
        # or whitening groups are attached per launch (run_device)
        self._K_dev, self._D_host = K, D
        self.problem = engine.SharedProblem(K, err if (shared and self.err is not None) else 1.0, D, omega.delta,
                                            variant=self.cost_function, reduce_singular_space=self.reduce_singular_space,
                                            device=dev, svd=self.svd, A_init=self.A_init)
        return self.problem

    def _group_problem(self, spec):
        """SharedProblem of one whitening group: the base kernel SVD with the group's error vector / covariance rotation,
        cached under the group's content."""
        import torch
        T, err = spec
        key = (None if T is None else T.tobytes(), err.tobytes())
        if key not in self._group_cache:
            base = self.prepare()
            K, U = self._K_dev, base.U
            if T is not None:
                Td = torch.as_tensor(T, device=base.device)
                K, U = Td @ K, Td @ U
            self._group_cache[key] = engine.SharedProblem(
                K, err, self._D_host, self.omega.delta, variant=self.cost_function, device=base.device, svd=self.svd,
                A_init=self.A_init, usv=(U, base.S, base.V), orthonormal_U=T is None)
        return self._group_cache[key]

    def alpha_effective(self):
        """alpha * scale_alpha (python/maxent_loop.py:216-232)."""
        a = np.asarray(self.alpha_mesh, dtype=np.float64)
        if self.scale_alpha is None:
            return a
        if isinstance(self.scale_alpha, str):
            if self.scale_alpha.lower() != "ndata":
                raise Exception("Unknown value {} for scale_alpha".format(self.scale_alpha))
            return a * self._n_data(self.prepare().n_tau)
        return a * float(self.scale_alpha)

    def run_device(self, G_dev, want_A=True, want_v=False, D=None, skip_small=False, v0=None):
        """Hot path on device-resident data: returns an engine.SweepResult of device tensors.
        ``D`` [B, n_omega] (optional): one default model per spectrum, incl. delta omega like ``DefaultModel.D``; with
        ``v0`` [B, n_sv] the model rows are ready-made (D [B, ldD], engine.run_sweep).
        Per-spectrum error models (set_error / set_cov with a leading batch axis) are applied here.
        ``skip_small``: spectra with max|G| < G_threshold are NOT continued (python/maxent_loop.py:174-179): they are left
        out of the launch and come back with status MX_STATUS_SKIPPED, NaN scalars, alpha_index -1 and A = 0.  For
        Matsubara data (stacked rows [Re G; Im G]) |G| is the complex modulus, as MaxEntLoop.run takes it."""
        import torch
        skip = skip_small and G_dev.dim() > 1
        G = G_dev if G_dev.dim() > 1 else G_dev[None, :]
        B = int(G.shape[0])
        plan = self._batch_plan(B)
        if skip and B:
            if self.iomega is not None:
                n_iw = G.shape[1] // 2
                small = torch.hypot(G[:, :n_iw], G[:, n_iw:]).amax(dim=1) < self.G_threshold
            else:
                small = G.abs().amax(dim=1) < self.G_threshold
            if bool(small.any()):
                keep = torch.nonzero(~small).flatten()
                kept = keep.cpu().numpy()
                Dk = None if D is None else (D[keep] if torch.is_tensor(D) else np.asarray(D)[kept])
                vk = None if v0 is None else v0[keep].contiguous()
                r = self._launch(plan.subset(kept), G[keep].contiguous(), want_A, want_v, Dk, vk) if len(kept) else None
                return self._scatter(r, keep, plan, B, want_A, want_v)
        return self._launch(plan, G, want_A, want_v, D, v0)

    def _launch(self, plan, G, want_A, want_v, D, v0):
        import torch
        if plan.rotations is not None:           # covariance groups: rotate the data, G' = T_g G
            Gr = torch.zeros((G.shape[0], max(q.n_tau for q in plan.problems)), dtype=torch.float64, device=G.device)
            for g, T in enumerate(plan.rotations):
                sel = torch.as_tensor(np.nonzero(plan.index == g)[0], device=G.device)
                if len(sel):
                    Gr[sel, :plan.problems[g].n_tau] = G[sel] @ torch.as_tensor(T, device=G.device).T
            G = Gr
        return engine.run_sweep(plan.problems[0], G, plan.alpha, probability=self.probability is not None,
                                lm=self.minimizer, want_A=want_A, want_v=want_v, gamma=self.gamma,
                                linefit_deg=self.linefit_deg, bryan_by_integration=self.bryan_by_integration, D=D, v0=v0,
                                sigma=plan.sigma, groups=None if plan.index is None else (plan.problems, plan.index),
                                alpha_scale=plan.alpha_scale)

    def _scatter(self, r, keep, plan, B, want_A, want_v):
        """The result `r` of the spectra `keep` of a batch of B, in full-size tensors; the other spectra come back
        skipped."""
        import torch
        prob = self.prepare()
        dev = prob.device
        n_alpha = len(self.alpha_mesh)
        full = engine.SweepResult()
        full.alpha = torch.as_tensor(self.alpha_effective(), device=dev) if r is None else r.alpha
        full.n_sv = prob.n_sv
        full.alpha_scale, full.problems, full.index = plan.alpha_scale, plan.problems, plan.index

        def blank(shape, dtype, fill):
            return torch.full((B,) + shape, fill, dtype=dtype, device=dev)
        f64, i32 = torch.float64, torch.int32
        spec = dict(chi2=((n_alpha,), f64, float("nan")), S=((n_alpha,), f64, float("nan")), Q=((n_alpha,), f64, float("nan")),
                    logp=((n_alpha,), f64, float("nan")), n_iter=((n_alpha,), i32, 0), n_qeval=((n_alpha,), i32, 0),
                    n_solve=((n_alpha,), i32, 0), status=((n_alpha,), i32, _lib.STATUS_SKIPPED), n_trial=((n_alpha,), i32, 0),
                    n_batch=((n_alpha,), i32, 0), alpha_index=((_lib.N_ANALYZERS,), i32, -1))
        for name, (shape, dtype, fill) in spec.items():
            t = blank(shape, dtype, fill)
            if r is not None and getattr(r, name) is not None:
                t[keep] = getattr(r, name)
            setattr(full, name, t)
        for name, shape in (("A", (n_alpha, prob.n_omega)), ("A_out", (_lib.N_ANALYZERS, prob.n_omega)), ("v", (n_alpha, prob.n_sv))):
            src = None if r is None else getattr(r, name)
            want = want_A if name != "v" else want_v
            if not want:
                setattr(full, name, None)
                continue
            t = blank(shape, f64, 0.0)
            if src is not None:
                t[keep] = src
            setattr(full, name, t)
        full.phase_cycles = None
        return full

    def time_sweep_kernel(self, G_dev):
        """Milliseconds of the mx_alpha_sweep launch alone (CUDA events on the launching stream)."""
        prob = self.prepare()
        return engine.run_sweep(prob, G_dev, self.alpha_effective(), probability=self.probability is not None,
                                lm=self.minimizer, want_A=True, want_v=False, time_kernel=True)

    def run(self, G=None, D=None):
        """Public call: host G[B, n_tau] in (numpy or pinned tensor), BatchedMaxEntResult (host arrays) out.
        ``D`` [B, n_omega] optionally gives every spectrum its own default model."""
        import torch
        G = self.G if G is None else G
        if G is None:
            raise Exception("no data: call set_G_tau_data or set_G_iw_data")
        if G.is_complex() if torch.is_tensor(G) else np.iscomplexobj(G):
            raise NotImplementedError("complex data: pass G(i omega_n) through set_G_iw_data")
        prob = self.prepare()
        dev = prob.device
        Gt = G if torch.is_tensor(G) else torch.from_numpy(np.ascontiguousarray(G, dtype=np.float64))
        if Gt.dim() == 1:
            Gt = Gt[None, :]
        out = BatchedMaxEntResult()
        out.h2d_bytes = Gt.numel() * 8 if not Gt.is_cuda else 0
        with torch.cuda.device(dev):
            G_dev = Gt.to(dev, non_blocking=True)
            # spectra below the threshold are not continued by the reference (maxent_loop.py:174-179): skip_small
            res = self.run_device(G_dev, D=D, skip_small=True)
            small = ((res.status[:, 0] & _lib.STATUS_SKIPPED) != 0) if G_dev.shape[0] else None
            host = {}
            n_d2h = 0
            for name, t in (("chi2", res.chi2), ("S", res.S), ("Q", res.Q), ("probability", res.logp),
                            ("n_iter", res.n_iter), ("status", res.status), ("alpha_index", res.alpha_index),
                            ("A_out", res.A_out), ("small", small)):
                if t is None:
                    host[name] = None
                    continue
                buf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
                buf.copy_(t, non_blocking=True)
                n_d2h += t.numel() * t.element_size()
                host[name] = buf
            torch.cuda.current_stream(dev).synchronize()
        out.d2h_bytes = n_d2h
        out.device = res
        out.omega = self.omega
        out.alpha = self.alpha_effective()
        for name in ("chi2", "S", "Q", "probability", "n_iter", "alpha_index", "A_out"):
            setattr(out, name, host[name].numpy())
        out.converged = (host["status"].numpy() & _lib.STATUS_CONVERGED).astype(bool)
        out.zero_elements = [] if host["small"] is None else np.nonzero(host["small"].numpy())[0].tolist()
        out.n_sv = prob.n_sv
        return out


def gather_results(out, dst=0):
    """The one collective of a multi-GPU job: gather the per-rank analyzer outputs on ``dst``
    (NCCL when the process group is nccl; gloo in the CPU tests).  Returns a dict of concatenated
    arrays on ``dst`` and None elsewhere."""
    import torch
    import torch.distributed as dist
    world, rank = dist.get_world_size(), dist.get_rank()
    backend = dist.get_backend()
    got = {}
    dev_res = getattr(out, "device", None)
    for name in ("alpha_index", "chi2", "A_out"):
        if backend == "nccl" and dev_res is not None and getattr(dev_res, name, None) is not None:
            t = getattr(dev_res, name).contiguous()          # results are still resident: no host round trip
        else:
            t = torch.as_tensor(np.ascontiguousarray(getattr(out, name)))
            if backend == "nccl":
                t = t.cuda()
        sizes = [torch.zeros(1, dtype=torch.int64, device=t.device) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([t.shape[0]], dtype=torch.int64, device=t.device))
        # the ranks' shards land in slices of ONE buffer on dst (no concatenation pass); the host copy goes into
        # pinned memory when the data is on a device (a pageable copy of the 2.6 GB of A_out of a 65,536-spectrum
        # job ran at ~3 GB/s and dominated the gather)
        counts = [int(n) for n in sizes]
        if rank == dst:
            full = torch.empty((sum(counts),) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
            parts = list(full.split(counts, 0)) if full.shape[0] else [full[:0] for _ in counts]
        else:
            full = parts = None

        def to_host(x):
            if not x.is_cuda:
                return x.numpy()
            h = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
            h.copy_(x, non_blocking=True)
            torch.cuda.current_stream(x.device).synchronize()
            return h.numpy()

        if all(n == counts[0] for n in counts):
            # equal shards (the benchmark's case): one gather collective
            dist.gather(t, parts, dst=dst)
            if rank == dst:
                got[name] = to_host(full)
            continue
        # ragged shards: point-to-point gather
        if rank == dst:
            for r in range(world):
                if r == dst:
                    parts[r].copy_(t)
                elif parts[r].numel():
                    dist.recv(parts[r], src=r)
            got[name] = to_host(full)
        elif t.numel():
            dist.send(t, dst=dst)
    return got if rank == dst else None
