/*
 * maxent_b200 -- C ABI of the B200-native MaxEnt alpha-sweep engine.
 *
 * The reference (TRIQS/maxent 1.2.0) is pure Python and has no FFI; the seam this library plugs
 * into is MaxEntLoop.run (python/maxent_loop.py:144-302) and the functions below it (SURVEY.md
 * section 8(a) R1-R13).  Each entry point names the reference code it replaces.
 *
 * Conventions: plain pointers and sizes, no torch / C++ types.  All pointers are DEVICE pointers
 * unless the name ends in _host.  Row-major contiguous float64 unless stated.  Every call is
 * asynchronous on `stream` (a cudaStream_t passed as void*), keeps no global state, and returns 0
 * or a negative MX_ERR_* code; nothing throws across the ABI.
 */
#ifndef MAXENT_B200_H
#define MAXENT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MX_OK                0
#define MX_ERR_BAD_ARG      -1
#define MX_ERR_UNSUPPORTED  -2   /* e.g. n_sv > MX_MAX_NSV */
#define MX_ERR_CUDA         -3
#define MX_ERR_NO_DEVICE    -4

#define MX_MAX_NSV         256   /* singular-space dimension the fused path supports: up to 80 with every matrix in
                                    * shared memory and registers, 81..256 with Z, J and the factors in the workspace */

/* sweep engines (MxProblem.engine) */
#define MX_ENGINE_AUTO       0   /* = MX_ENGINE_SPECTRUM_CTA */
#define MX_ENGINE_LOCKSTEP   1   /* retired (round-1 lock-step engine): requesting it returns MX_ERR_UNSUPPORTED */
#define MX_ENGINE_SPECTRUM_CTA 2 /* one spectrum per CTA, speculative damping batches (csrc/mx_sweep2.cuh)    */

/* MxProblem.per_spectrum_model bits */
#define MX_PER_SPECTRUM_MODEL 1
#define MX_PER_SPECTRUM_XI    2
#define MX_PER_SPECTRUM_VT    4
#define MX_PER_SPECTRUM_ALPHA 8

/* cost-function variants (python/maxent_loop.py:106-121) */
#define MX_VARIANT_NORMAL    0   /* MaxEntCostFunction + NormalEntropy + NormalH_of_v   */
#define MX_VARIANT_PLUSMINUS 1   /* MaxEntCostFunction + PlusMinusEntropy + PlusMinusH_of_v */
#define MX_VARIANT_BRYAN     2   /* BryanCostFunction */

/* analyzer slots in mx_analyze outputs */
#define MX_AN_LINEFIT        0   /* python/analyzers/linefit_analyzer.py        */
#define MX_AN_CHI2CURV       1   /* python/analyzers/chi2_curvature_analyzer.py */
#define MX_AN_ENTROPY        2   /* python/analyzers/entropy_analyzer.py        */
#define MX_AN_CLASSIC        3   /* python/analyzers/classic_analyzer.py        */
#define MX_AN_BRYAN          4   /* python/analyzers/bryan_analyzer.py          */
#define MX_N_ANALYZERS       5

/* per-(spectrum, alpha) status bits */
#define MX_STATUS_CONVERGED  1   /* LevenbergMinimizer.converged (levenberg_minimizer.py:162-174) */
#define MX_STATUS_SKIPPED    2   /* max|G| < G_threshold (maxent_loop.py:174-179): set by the host front end, which
                                  * leaves such spectra out of the launch (maxent_b200/batched.py) */

/* Levenberg-Marquardt parameters = LevenbergMinimizer.__init__ (levenberg_minimizer.py:92-121)
 * with the default convergence MaxDerivative(1e-4) | RelativeFunctionChange(1e-16); a criterion is switched off
 * by a negative threshold.  J_squared is not available. */
typedef struct {
    int32_t maxiter;          /* 1000  */
    int32_t miniter;          /* 0     */
    double  mu0;              /* 1e-18 */
    double  nu;               /* 1.3   */
    double  max_mu;           /* 1e20  */
    double  conv_max_derivative;   /* 1e-4  */
    double  conv_rel_change;       /* 1e-16 */
    double  conv_abs_change;       /* -1 (off): FunctionChangeConvergenceMethod, |Q0 - Q1| < x (convergence_methods.py:100-110) */
    int32_t marquardt;             /* 0: J + mu 1 ; 1: J + mu diag(J)   (levenberg_minimizer.py:181-185) */
    int32_t reserved;              /* 0 */
} MxLMParams;

/* Problem state shared by every spectrum of a batch (built once per kernel/err by
 * mx_layout_V + the host-side preparation; see DESIGN.md "data layout"). */
typedef struct {
    int32_t n_tau;            /* rows of the (possibly covariance-rotated) data space       */
    int32_t n_omega;
    int32_t n_sv;             /* singular-space dimension s  (<= MX_MAX_NSV)                 */
    int32_t n_alpha;
    int32_t variant;          /* MX_VARIANT_*                                                */
    int32_t want_probability; /* NormalLogProbability (probabilities.py:76-85)               */
    int32_t engine;           /* MX_ENGINE_*                                                 */
    int32_t per_spectrum_model; /* bit mask.  MX_PER_SPECTRUM_MODEL: D[B, ldD], v0[B, n_sv] instead of D[n_omega], v0[n_sv],
                               * row stride ldD = n_omega rounded up to an even number (16-byte aligned rows)
                               * (PoormanMaxEnt off-diagonals, python/elementwise_maxent.py:633-652).
                               * MX_PER_SPECTRUM_XI: xi[B, n_sv] instead of xi[n_sv] -- every spectrum carries its own
                               * scalar error bar, Xi_b = S / sigma_b (TauMaxEnt.set_error per data set,
                               * python/tau_maxent.py:227-251); G is then passed already divided by sigma_b.
                               * MX_PER_SPECTRUM_VT: spectra belong to groups with different error vectors / covariances,
                               * i.e. different whitening rotations: see vt_index (xi, D, v0 per spectrum as well).
                               * MX_PER_SPECTRUM_ALPHA: alpha[B, n_alpha] -- scale_alpha = 'Ndata' multiplies alpha by the
                               * number of data rows (python/maxent_loop.py:216-220), which differs between groups whose
                               * covariance matrices drop different numbers of eigenvalues */
    double  chi2_factor;      /* MaxEntCostFunction chi2_factor (cost_function.py:43-53)     */
    const double* Vt;         /* swizzled tile-major V' written by mx_layout_V               */
    const double* Qw;         /* [n_tau, n_sv]  sqrt(W) Q : g~ = Qw^T G                      */
    const double* Qo;         /* [n_tau, n_sv]  Q (orthonormal) for the out-of-range residual */
    const double* sqrtw;      /* [n_tau]        1/err                                         */
    const double* xi;         /* [n_sv]         singular values of sqrt(W) K V_s             */
    const double* D;          /* [n_omega] or [B, n_omega]  default model incl. delta omega  */
    const double* delta;      /* [n_omega]      trapezoid weights of the omega mesh          */
    const double* alpha;      /* [n_alpha]      alpha * scale_alpha, descending              */
    const double* v0;         /* [n_sv] or [B, n_sv]  initial v' (maxent_loop.py:196-203)    */
    MxLMParams lm;
    const int32_t* vt_index;  /* MX_PER_SPECTRUM_VT: [B] index of the spectrum's whitening group; its V' starts at
                               * Vt + vt_index[b] * vt_stride (every group: its own rotation V' = V_s P_g, python/tau_maxent.py:
                               * 227-288 per data set); NULL otherwise */
    int64_t vt_stride;        /* doubles between the V' buffers of consecutive groups (>= mx_layout_V_size) */
} MxProblem;

/* Outputs of the alpha sweep; any pointer may be NULL to skip that output (chi2/S/Q required). */
typedef struct {
    double*  v;        /* [B, n_alpha, n_sv]     solution in the (rotated) singular basis  */
    double*  A;        /* [B, n_alpha, n_omega]  A_alpha(omega) = H / delta (functions.py:947-952) */
    double*  chi2;     /* [B, n_alpha]   */
    double*  S;        /* [B, n_alpha]   */
    double*  Q;        /* [B, n_alpha]   */
    double*  logp;     /* [B, n_alpha]   NaN if !want_probability */
    int32_t* n_iter;   /* [B, n_alpha]   LevenbergMinimizer.n_iter_last */
    int32_t* n_qeval;  /* [B, n_alpha]   cost-function evaluations (rounds) */
    int32_t* n_solve;  /* [B, n_alpha]   dense solves attempted */
    int32_t* status;   /* [B, n_alpha]   MX_STATUS_* bits */
    int32_t* n_trial;  /* [B, n_alpha]   trial points the device evaluated (incl. mis-speculated ones); may be NULL */
    int32_t* n_batch;  /* [B, n_alpha]   speculative batches (= passes over V' for cost evaluations); may be NULL */
    int64_t* phase_cycles; /* [B, 8]     SM clock cycles per spectrum spent in: planner, solver, T-pass, H-pass, gradient,
                            *             J assembly, other (accept, convergence test, outputs), replay of the damping
                            *             search on the tabulated trials (diagnostics; may be NULL)                     */
} MxSweepOut;

/* Library / device info.  Returns the number of SMs of the current device (or <0). */
int mx_device_sm_count(void);
const char* mx_version(void);

/* Measurement helper (bench.py): achieved FP64 TFLOP/s of the current device with every SM saturated by independent
 * DMMA (mma.sync m8n8k4 f64) and by DFMA chains -- the roofline denominator of the sweep kernel, measured inside the
 * benchmark run.  `scratch` = device buffer of at least 2 * SMs * 256 doubles.  Synchronous (returns host numbers). */
int mx_fp64_peak(double* tflops_dmma_host, double* tflops_dfma_host, double* scratch, void* stream);

/* Size in doubles of the swizzled V buffer for (n_omega, n_sv). */
int64_t mx_layout_V_size(int32_t n_omega, int32_t n_sv);

/* Re-tile V [n_omega, n_sv] (row-major) into the bank-conflict-free 8x8 tile layout the sweep
 * kernel streams.  Replaces nothing in the reference (layout only). */
int mx_layout_V(const double* V, int32_t n_omega, int32_t n_sv, double* Vt, void* stream);

/* TauKernel._fill_values (python/kernels.py:244-266): K[n_tau, n_omega] on the device. */
int mx_tau_kernel(const double* tau, const double* omega, int32_t n_tau, int32_t n_omega,
                  double beta, double* K, void* stream);

/* One-sided (Hestenes) Jacobi SVD of K[m, n] (m >= n), every column: replaces np.linalg.svd in KernelSVD.svd
 * (python/kernels.py:53-64).  U[m, n], S[n] (descending), V[n, n]; work = m*n + n*n + n + 64 doubles.  One persistent
 * cooperative kernel, convergence decided on the device; `sweeps_done` (host, may be NULL) is filled by a
 * stream-ordered copy, i.e. valid once the caller has synchronised `stream`. */
int mx_svd_jacobi(const double* K, int32_t m, int32_t n, double* U, double* S, double* V,
                  double* work, int32_t max_sweeps, int32_t* sweeps_done, void* stream);

/* Truncated SVD: the leading p triplets of K[m, n] (any shape, p <= min(m, n)) by a random range finder followed by
 * one-sided Jacobi on p columns (csrc/mx_svd.cu).  U[m, p], S[p] (descending), V[n, p].  Exact to rounding
 * (|K - U S V^T| ~ eps * S[0]) whenever S[p-1] is at the rounding floor of K, i.e. whenever p exceeds the numerical rank:
 * the caller checks S[p-1] <= ~1e-15 * S[0] and asks again with a larger p otherwise.  Only triplets above the
 * caller's cut enter the MaxEnt loop (python/kernels.py:101-122).  work = mx_svd_truncated_work_doubles(m, n, p). */
int64_t mx_svd_truncated_work_doubles(int32_t m, int32_t n, int32_t p);
int mx_svd_truncated(const double* K, int32_t m, int32_t n, int32_t p, double* U, double* S, double* V,
                     double* work, uint64_t seed, void* stream);

/* Orthonormalise the p rows of Yt[p, len] in place, in order (classical Gram-Schmidt, every row projected three times
 * against the finished ones, one CTA; p <= 512).  A row whose residual falls below drop_rel times its norm is zeroed
 * (drop_rel = 0: never).  Used for Q = the left vectors of the whitened kernel, whose orthogonality chi2 relies on
 * (python/functions.py:358-360 evaluates chi2 with the full kernel and needs no such step). */
int mx_gram_schmidt_rows(double* Yt, int32_t len, int32_t p, double drop_rel, void* stream);

/* Project the data of B spectra into the singular space:
 *   gt[b] = Qw^T G[b]  and  c0[b] = | sqrtw*G[b] - Qo gt[b] |^2
 * so that chi2(H) = sum_i (xi_i y_i - gt_i)^2 + c0 with y = V'^T H   (NormalChi2.f, functions.py:358-360). */
int mx_project_data(const MxProblem* p, const double* G /*[B, n_tau]*/, int32_t B,
                    double* gt /*[B, n_sv]*/, double* c0 /*[B]*/, void* stream);

/* The fused alpha sweep = the `for alpha in alpha_mesh` loop of MaxEntLoop.run
 * (python/maxent_loop.py:241-266) with LevenbergMinimizer.minimize
 * (python/minimizers/levenberg_minimizer.py:123-248), the cost functions
 * (python/cost_functions/maxent_cost_function.py:68-165, bryan_cost_function.py:57-128) and
 * NormalLogProbability.f (python/probabilities.py:76-85) for B independent spectra.
 * `workspace` is device memory of at least mx_sweep_workspace_bytes(p, B) bytes, 256-byte aligned
 * (work counter + per-CTA scratch rows); its contents need not be initialised.  */
int mx_alpha_sweep(const MxProblem* p, const double* gt, const double* c0, int32_t B,
                   const MxSweepOut* out, void* workspace, int64_t workspace_bytes, void* stream);

/* Device workspace mx_alpha_sweep needs for this problem and batch size on the current device (<0: MX_ERR_*). */
int64_t mx_sweep_workspace_bytes(const MxProblem* p, int32_t B);

/* Introspection for tests / DESIGN.md: engine actually used for (n_sv, engine), spectra marched per CTA,
 * dynamic shared memory and threads per CTA.  Needs no device. */
int mx_sweep_config(int32_t n_sv, int32_t engine, int32_t* engine_used, int32_t* spectra_per_cta,
                    int32_t* smem_bytes, int32_t* threads);

/* Analyzer reductions (python/analyzers/*.py) for B spectra:
 * alpha_index[B, MX_N_ANALYZERS] (-1 = not available), A_out[B, MX_N_ANALYZERS, n_omega] (may be NULL),
 * aux[B, 4 + 2 n_alpha] (may be NULL): the line-fit parameters {slope1, intercept1, slope2, intercept2}
 * (linefit_analyzer.py:63-69), curvature[n_alpha] (chi2_curvature_analyzer.py:25-49) and
 * dS/dlog(alpha)[n_alpha] (entropy_analyzer.py:92-95); entries that do not exist are NaN. */
int mx_analyze(const double* alpha /*[n_alpha]*/, const double* chi2, const double* S,
               const double* logp /* may be NULL */, const double* A /*[B, n_alpha, n_omega]*/,
               int32_t B, int32_t n_alpha, int32_t n_omega, double gamma, int32_t linefit_deg,
               int32_t bryan_by_integration,
               int32_t* alpha_index, double* A_out, double* aux, void* stream);

/* PoormanMaxEnt off-diagonal default models (python/elementwise_maxent.py:633-652) for P off-diagonal spectra, read from
 * the analyzer output of the diagonal pass (A_out of mx_analyze, R spectra) without a trip to the host:
 *   D[p]  = (sqrt(A_out[rows[2p], slot] * A_out[rows[2p+1], slot]) + d_add) * delta  (DataDefaultModel(...).D), rows of
 *           ldD = n_omega rounded up to an even number, padding zeroed (the layout of MX_PER_SPECTRUM_MODEL);
 *   v0[p] = V'^T log(arg), arg = (H0 + sqrt(H0^2 + 4 D^2)) / (2 D), H0 = (A_init or D[p]) * delta (maxent_loop.py:
 *           196-203), |arg| <= 1e-100 -> 1e-100; V' = Vp + group[p] * n_omega * n_sv (Vp[G, n_omega, n_sv], group may
 *           be NULL: G = 1).  Summed over omega in index order: independent of P and of p's position in the batch;
 *   ok[p] = 0 when either diagonal row holds a NaN (analyzer unavailable, element not continued), else 1.
 * The caller guarantees 0 <= rows < R and 0 <= group < G. */
int mx_poorman_models(const double* A_out /*[R, MX_N_ANALYZERS, n_omega]*/, int32_t slot, const int32_t* rows /*[P, 2]*/,
                      int32_t P, const double* delta, double d_add, const double* A_init /*[n_omega] or NULL*/,
                      const double* Vp, const int32_t* group /*[P] or NULL*/, int32_t n_omega, int32_t n_sv,
                      double* D /*[P, ldD]*/, double* v0 /*[P, n_sv]*/, int32_t* ok /*[P]*/, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MAXENT_B200_H */
