"""Pin the CPU oracle (oracle/maxent_oracle.py) against fixtures produced by the REAL reference
(tests/golden/*.npz, written by oracle/make_golden.py) and against the reference's own
known-answer numbers (test/python/tau_maxent.py:134-135).  CPU only."""
import os

import numpy as np
import pytest
import threadpoolctl

from oracle import maxent_oracle as mo

# oracle/make_golden.py wrote the fixtures on a host whose OpenBLAS ran its SkylakeX (AVX-512) kernels on 8 threads.
# How OpenBLAS splits a matrix product over its threads changes the last bits of the result, so the bit-identical
# comparisons below run on that many BLAS threads, whatever the number of cores of the host running the tests.
GOLDEN_BLAS_THREADS = 8


@pytest.fixture(scope="module", autouse=True)
def _golden_blas_threads():
    with threadpoolctl.threadpool_limits(limits=GOLDEN_BLAS_THREADS, user_api="blas"):
        yield


def _load(golden_dir, name):
    with np.load(os.path.join(golden_dir, name), allow_pickle=False) as z:
        return {k: z[k] for k in z.files}


def _run(g, **kw):
    beta = None
    K = mo.tau_kernel(g["tau"], g["omega"], beta)
    return mo.maxent_loop(K, g["G"], g["err"], g["omega"], g["alpha_mesh"], variant=str(g["variant"]),
                          probability=bool(g["use_probability"]),
                          reduce_singular_space=float(g["reduce_singular_space"]), **kw)


def _check_identical(out, g, fields=("chi2", "S", "Q", "A"), rtol=0.0):
    assert out["n_sv"] == int(g["ref_n_sv"])
    np.testing.assert_array_equal(out["alpha"], g["ref_alpha"])
    for f in fields:
        ref = g["ref_" + f]
        if rtol == 0.0:
            np.testing.assert_array_equal(out[f], ref, err_msg=f)
        else:
            np.testing.assert_allclose(out[f], ref, rtol=rtol, atol=rtol * np.max(np.abs(ref)), err_msg=f)
    for name, res in out["analyzers"].items():
        key = "ref_idx_" + name
        if key in g:
            assert res["alpha_index"] == int(g[key]), name
            np.testing.assert_array_equal(res["A_out"], g["ref_Aout_" + name])


def test_known_answer_probability(golden_dir):
    """test/python/tau_maxent.py:134-135 : the reference's literal probability values (6 decimals)."""
    g = _load(golden_dir, "g1_semicircular_prob.npz")
    out = _run(g)
    np.testing.assert_almost_equal(out["probability"], g["known_probability"], 6)
    _check_identical(out, g, fields=("chi2", "S", "Q", "A", "H", "probability"))
    # Bryan analyzer output is a weighted sum
    np.testing.assert_array_equal(out["analyzers"]["BryanAnalyzer"]["A_out"], g["ref_Aout_BryanAnalyzer"])


def test_synthetic_normal_bit_identical(golden_dir):
    g = _load(golden_dir, "g2_synth_200x100.npz")
    out = _run(g)
    _check_identical(out, g, fields=("chi2", "S", "Q", "A", "H", "probability"))


def test_plusminus_bit_identical(golden_dir):
    g = _load(golden_dir, "g3_plusminus_offdiag.npz")
    out = _run(g)
    _check_identical(out, g, fields=("chi2", "S", "Q", "A", "H"))


def test_bryan_bit_identical(golden_dir):
    g = _load(golden_dir, "g4_bryan_200x100.npz")
    out = _run(g)
    _check_identical(out, g, fields=("chi2", "S", "Q", "A", "H"))


def test_marquardt_and_function_change_bit_identical(golden_dir):
    """LevenbergMinimizer(marquardt=True, convergence=MaxDerivative(1e-4) | FunctionChange(1e-9)) run by the real
    reference (python/minimizers/levenberg_minimizer.py:181-185, convergence_methods.py:100-110)."""
    g = _load(golden_dir, "g8_marquardt_200x100.npz")
    out = _run(g, lm_options=dict(marquardt=bool(g["lm_marquardt"]), abs_change=float(g["lm_abs_change"])))
    _check_identical(out, g, fields=("chi2", "S", "Q", "A", "H"))
    base = _load(golden_dir, "g2_synth_200x100.npz")           # same data, default minimiser: a different path
    assert not np.array_equal(g["ref_chi2"], base["ref_chi2"])


def test_full_covariance_bit_identical(golden_dir):
    """TauMaxEnt.set_cov with a correlated covariance matrix run by the real reference (python/tau_maxent.py:253-288):
    eigenbasis rotation T, K' = T K, G' = T G, err = sqrt(eigenvalues); the SVD stays that of the unrotated kernel
    with U' = T U (python/kernels.py:160-180)."""
    g = _load(golden_dir, "g9_covariance_200x100.npz")
    K = mo.tau_kernel(g["tau"], g["omega"], None)
    e, v = np.linalg.eigh(g["cov"])
    keep = e >= 1.e-14                                     # cov_threshold default (python/tau_maxent.py:56)
    e, T = e[keep], v[:, keep].conjugate().transpose()
    np.testing.assert_array_equal(np.sqrt(e), g["err"])
    np.testing.assert_array_equal(np.dot(T, g["G"]), g["ref_G_rotated"])
    np.testing.assert_array_equal(np.dot(T, K)[0], g["ref_K_rotated_row0"])
    U, S, V = mo.kernel_svd(K, float(g["reduce_singular_space"]))
    out = mo.maxent_loop(np.dot(T, K), np.dot(T, g["G"]), np.sqrt(e), g["omega"], g["alpha_mesh"],
                         reduce_singular_space=float(g["reduce_singular_space"]), svd=(np.dot(T, U), S, V))
    _check_identical(out, g, fields=("chi2", "S", "Q", "A", "H"))


@pytest.mark.parametrize("name", ["g5_config1_cut1e-11.npz", "g5b_config1_default_cut.npz"])
def test_config1_bit_identical(golden_dir, name):
    """BASELINE config 1 (n_tau=1000, n_omega=400, 60 alphas): LineFit 23 / Chi2Curv 28 / Entropy 42."""
    g = _load(golden_dir, name)
    out = _run(g)
    _check_identical(out, g)
    assert out["analyzers"]["LineFitAnalyzer"]["alpha_index"] == 23
    assert out["analyzers"]["Chi2CurvatureAnalyzer"]["alpha_index"] == 28
    assert out["analyzers"]["EntropyAnalyzer"]["alpha_index"] == 42


def test_low_temperature_kernel_bit_identical(golden_dir):
    """beta = 1000: the reference keeps 82 singular values at its default cut -- the oracle for the wide
    instantiations of the sweep kernel (n_sv > 80)."""
    g = _load(golden_dir, "g15_low_temperature_wide.npz")
    out = _run(g)
    assert out["n_sv"] == int(g["ref_n_sv"]) == 82
    _check_identical(out, g)
    assert out["analyzers"]["LineFitAnalyzer"]["alpha_index"] == int(g["ref_idx_LineFitAnalyzer"]) == 14
    assert out["analyzers"]["Chi2CurvatureAnalyzer"]["alpha_index"] == int(g["ref_idx_Chi2CurvatureAnalyzer"]) == 17


def test_meshes_and_kernel():
    """test/python/tau_kernel.py:27-69 : independent kernel formula to 1e-15; U S V^T reconstructs K."""
    tau = np.linspace(0, 10, 50)
    om = mo.hyperbolic_omega_mesh(-5, 5, 30)
    K = mo.tau_kernel(tau, om, 10.0)
    Kind = np.array([[-np.exp(-t * w) / (1 + np.exp(-10.0 * w)) if w >= 0 else
                      -np.exp((10.0 - t) * w) / (1 + np.exp(10.0 * w)) for w in om] for t in tau])
    assert np.max(np.abs(K - Kind)) < 1e-15
    U, S, V = mo.kernel_svd(K, None)
    assert np.max(np.abs(np.dot(U * S, V.T) - K)) < 1e-13
    U2, S2, V2 = mo.kernel_svd(K, np.median(S))
    assert len(S2) == (len(S) + 1) // 2
    d = mo.omega_delta(om)
    assert abs(np.sum(d) - 10.0) < 1e-13
    D = mo.flat_default_model(om)
    assert abs(np.sum(D) - 1.0) < 1e-14
    a = mo.log_alpha_mesh(0.01, 2000, 60)
    assert a[0] > a[-1] and abs(a[0] - 2000) < 1e-9 and abs(a[-1] - 0.01) < 1e-12
