"""Helpers shared by the `-m gpu` parity tests: run a fixture through the C ABI (via the ctypes
host engine) and compare with reference / oracle outputs under the tiered contract of
SURVEY.md section 8(c)."""
import os

import numpy as np

from oracle import maxent_oracle as mo

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
AN_NAMES = ("LineFitAnalyzer", "Chi2CurvatureAnalyzer", "EntropyAnalyzer", "ClassicAnalyzer", "BryanAnalyzer")

# --- the parity contract (floating point; SURVEY.md 8(c)) --------------------------------------
RTOL_WELL_DETERMINED = 1.e-8      # T2: A (max-norm relative), chi2, S, Q where the reference reproduces itself
NOISE_FACTOR = 10.0               # T4: elsewhere, 10x the reference's own noise floor (fixture field noise_*)
PROB_RTOL = 1.e-6                 # probability: abs error <= 1e-6 * |p|


def load_golden(name):
    with np.load(os.path.join(GOLDEN, name), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def running_max(x, half=2):
    x = np.asarray(x, dtype=float)
    return np.array([np.max(x[max(0, i - half):i + half + 1]) for i in range(len(x))])


# rounding-level perturbations of the data used to measure the oracle's own noise floor where it is run live
EPS = (1e-15, -1e-15, 2e-15, -2e-15)


def oracle_floor(base, run):
    """Noise floor of a live oracle result `base`: the largest movement of A and chi2, per alpha, over the runs
    run(1 + eps) for the rounding-level perturbations EPS (one sample is a noisy estimate of the floor, and the small-alpha
    tail amplifies rounding differences by many orders of magnitude).  Returns (noise_A, noise_chi2), running maxima
    over +-2 alphas."""
    nA = np.zeros(len(base["chi2"]))
    nc = np.zeros(len(base["chi2"]))
    for e in EPS:
        o2 = run(1.0 + e)
        nA = np.maximum(nA, rel_A(o2["A"], base["A"]))
        nc = np.maximum(nc, np.abs(o2["chi2"] / base["chi2"] - 1))
    return running_max(nA), running_max(nc)


def tolerances(g, field):
    """Per-alpha tolerance: 1e-8 where the reference is reproducible to better than that, else
    10x its own measured noise floor (running max over +-2 alphas: one sample is a noisy estimate)."""
    noise = running_max(g["noise_" + field])
    return np.maximum(RTOL_WELL_DETERMINED, NOISE_FACTOR * noise)


def run_fixture(g, svd="jacobi", B=1, **kw):
    """Fused GPU sweep on the inputs of a golden fixture; returns (SharedProblem, SweepResult)."""
    from maxent_b200 import engine
    K = mo.tau_kernel(g["tau"], g["omega"], None)
    delta = mo.omega_delta(g["omega"])
    D = mo.flat_default_model(g["omega"])
    prob = engine.SharedProblem(K, g["err"], D, delta, variant=str(g["variant"]),
                                reduce_singular_space=float(g["reduce_singular_space"]), svd=svd)
    G = np.repeat(np.asarray(g["G"])[None, :], B, axis=0)
    res = engine.run_sweep(prob, G, g["ref_alpha"], probability=bool(g["use_probability"]), **kw)
    return prob, res


def sweep_tiles(n_sv):
    """Tile count NT of the sweep instantiation for n_sv (sweep_tiles in mx_common.cuh): 8 columns per tile, at least
    4, multiples of 4 above 10 (the wide instantiations)."""
    nt = max((n_sv + 7) // 8, 4)
    return (nt + 3) & ~3 if nt > 10 else nt


def kernel_problem(n_sv, n_tau, n_om, variant, seed, n_spectra):
    """A DataKernel K = U diag(logspace(0, -6, n_sv)) V^T plus a floor of 1e-14, with exactly n_sv singular values above
    the cut 1e-9 (the construction of test_gpu_parity; n_tau >= n_om), and n_spectra noisy data sets of a two-peak
    spectrum (plus-minus: with a negative lobe).  Returns (K, G, omega, delta)."""
    rng = np.random.RandomState(seed)
    om = mo.linear_omega_mesh(-4, 4, n_om)
    U, _ = np.linalg.qr(rng.randn(n_tau, n_om))
    V, _ = np.linalg.qr(rng.randn(n_om, n_om))
    S = np.concatenate([np.logspace(0, -6, n_sv), 1e-14 * np.ones(n_om - n_sv)])
    K = (U * S) @ V.T
    A_true = np.exp(-(om - 0.5) ** 2) + 0.5 * np.exp(-(om + 1.5) ** 2 / 0.5)
    if variant == "plusminus":
        A_true = A_true - 0.8 * np.exp(-(om - 2.0) ** 2 / 0.3)
    delta = mo.omega_delta(om)
    G = (K * delta[None, :]) @ A_true + 1e-4 * rng.randn(n_spectra, n_tau)
    return K, G, om, delta


def rel_A(A, Aref):
    return np.max(np.abs(A - Aref), axis=-1) / np.max(np.abs(Aref), axis=-1)


def check_against_reference(g, res, b=0, rtol_chi2_S=RTOL_WELL_DETERMINED):
    """Tiers T2-T4 against the reference outputs stored in the fixture.  ``rtol_chi2_S`` is the floor for
    chi2 and S separately (Q and A keep 1e-8): when the kernel matrix itself comes from another exp()
    implementation (device TauKernel, 1 ulp) the Levenberg path may stop at a different point inside the
    reference's own convergence ball (max|dQ/dv| < 1e-4); Q is stationary there (second-order error) but chi2
    and S move at first order, in opposite directions."""
    A = res.A[b].cpu().numpy()
    chi2 = res.chi2[b].cpu().numpy()
    S = res.S[b].cpu().numpy()
    Q = res.Q[b].cpu().numpy()
    tolA, tolc, tolS = tolerances(g, "A"), tolerances(g, "chi2"), tolerances(g, "S")
    tolQ = np.maximum(tolc, tolS)
    tolc, tolS = np.maximum(tolc, rtol_chi2_S), np.maximum(tolS, rtol_chi2_S)
    dA = rel_A(A, g["ref_A"])
    assert np.all(dA <= tolA), "A: worst ratio %.2f at alpha idx %d" % (np.max(dA / tolA), int(np.argmax(dA / tolA)))
    dc = np.abs(chi2 / g["ref_chi2"] - 1)
    assert np.all(dc <= tolc), "chi2: worst ratio %.2f at %d" % (np.max(dc / tolc), int(np.argmax(dc / tolc)))
    dS = np.abs(S / g["ref_S"] - 1)
    assert np.all(dS <= np.maximum(tolS, tolA)), "S: %s" % (dS / np.maximum(tolS, tolA),)
    dQ = np.abs(Q / g["ref_Q"] - 1)
    assert np.all(dQ <= tolQ), "Q: %s" % (dQ,)
    if bool(g["use_probability"]):
        p = res.logp[b].cpu().numpy()
        ptol = np.maximum(PROB_RTOL, NOISE_FACTOR * running_max(g["noise_chi2"]))
        assert np.all(np.abs(p - g["ref_probability"]) <= ptol * np.abs(g["ref_probability"])), (p, g["ref_probability"])
    # T3: decisions
    idx = res.alpha_index[b].cpu().numpy()
    Aout = res.A_out[b].cpu().numpy()
    for slot, name in enumerate(AN_NAMES[:4]):
        key = "ref_idx_" + name
        if key in g:
            assert idx[slot] == int(g[key]), "%s picked %d, reference %d" % (name, idx[slot], int(g[key]))
            ref = g["ref_Aout_" + name]
            assert np.max(np.abs(Aout[slot] - ref)) <= tolA[idx[slot]] * np.max(np.abs(ref)), name
        else:
            assert idx[slot] == -1, name
    if "ref_Aout_BryanAnalyzer" in g:
        # Bryan averages A_alpha with weights exp(p - max p): its tolerance is the weighted tolerance of the
        # spectra it averages (the weights can sit on the noisy small-alpha tail), floor 1e-6 (SURVEY.md 8(c) T3)
        ref = g["ref_Aout_BryanAnalyzer"]
        w = np.exp(g["ref_probability"] - np.nanmax(g["ref_probability"]))
        w = np.where(np.isnan(w), 0.0, w) / np.nansum(w)
        btol = max(1.e-6, float(np.sum(w * tolA) * 2))
        assert np.max(np.abs(Aout[4] - ref)) <= btol * np.max(np.abs(ref)), (np.max(np.abs(Aout[4] - ref)), btol)
    return dict(dA=dA, dchi2=dc)


def check_matrix_result(res, g, hermitian_copy=()):
    """The tiered contract (T2-T4) element by element for the matrix front ends (ElementwiseMaxEnt, PoormanMaxEnt, with
    or without complex elements) against a run of the real reference: A and chi2 within 1e-8 where the reference
    reproduces itself, 10x its own noise floor elsewhere; LineFit picks identical; A_out at the tolerance of the pick.
    Elements the reference did not compute (NaN) must be NaN here too."""
    refA, refc = g["ref_A"], g["ref_chi2"]
    A, chi2 = np.asarray(res.A), np.asarray(res.chi2)
    assert A.shape == refA.shape and chi2.shape == refc.shape, (A.shape, refA.shape)
    worst = 0.0
    for el in np.ndindex(*refc.shape[:-1]):
        if np.all(np.isnan(refc[el])):
            assert np.all(np.isnan(chi2[el])), el
            continue
        tolA = np.maximum(RTOL_WELL_DETERMINED, NOISE_FACTOR * running_max(np.nan_to_num(g["noise_A"][el])))
        tolc = np.maximum(RTOL_WELL_DETERMINED, NOISE_FACTOR * running_max(np.nan_to_num(g["noise_chi2"][el])))
        dA = rel_A(A[el], refA[el])
        assert np.all(dA <= tolA), (el, dA / tolA)
        dc = np.abs(chi2[el] / refc[el] - 1.0)
        assert np.all(dc <= tolc), (el, dc / tolc)
        worst = max(worst, float(np.max(dA / tolA)))
        ij, c = el[:2], (el[2] if len(el) > 2 else 0)
        k = int(g["ref_idx_LineFitAnalyzer"][ij[0], ij[1], c])
        ar = res.analyzer_results[ij[0]][ij[1]]
        ar = ar[c] if isinstance(ar, (list, tuple)) else ar
        assert int(ar["LineFitAnalyzer"]["alpha_index"]) == k, (el, ar["LineFitAnalyzer"]["alpha_index"], k)
        ref_out = refA[el][k]
        assert np.max(np.abs(np.asarray(ar["LineFitAnalyzer"]["A_out"]) - ref_out)) <= tolA[k] * np.max(np.abs(ref_out)), el
    ro, mo_ = g["ref_A_out"], np.asarray(res.A_out)
    assert np.array_equal(np.isnan(ro), np.isnan(mo_))
    assert np.nanmax(np.abs(mo_ - ro)) <= 1e-7 * np.nanmax(np.abs(ro))
    return worst
