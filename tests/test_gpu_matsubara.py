"""GPU tests of Matsubara data in BatchedTauMaxEnt: the device fill of the IOmegaKernel, the batch against the run of
the real reference (fixture g14) and against the single-spectrum MaxEntLoop row by row, per-spectrum error models in one
launch, and the threshold skip on the complex modulus."""
import ctypes

import numpy as np
import pytest

import maxent_b200 as mb
from tests import gpu_common as gc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _batch(g, B, seed=11):
    """g14's G as row 0, the other rows g14's G with fresh noise of the fixture's error bar."""
    rng = np.random.default_rng(seed)
    G = np.repeat(g["G"][None, :], B, axis=0)
    G[1:] += float(g["err"]) * (rng.standard_normal((B - 1, len(g["G"]))) + 1j * rng.standard_normal((B - 1, len(g["G"]))))
    return G


def _job(g, **kw):
    j = mb.BatchedTauMaxEnt(reduce_singular_space=float(g["reduce_singular_space"]), probability="normal", **kw)
    j.omega = mb.DataOmegaMesh(g["omega"])
    j.alpha_mesh = mb.DataAlphaMesh(g["alpha_mesh"])
    return j


@pytest.mark.parametrize("mesh", ["g14", "hyperbolic_with_zero"])
def test_iomega_kernel_fill(torch_cuda, mesh):
    """mx_iomega_kernel = IOmegaKernel(iomega, omega).fused_matrix() (numpy's complex division) to rtol 1e-15."""
    torch = torch_cuda
    from maxent_b200 import _lib
    g = gc.load_golden("g14_iomega_200x100.npz")
    om = mb.DataOmegaMesh(g["omega"]) if mesh == "g14" else mb.DataOmegaMesh(np.concatenate([
        np.asarray(mb.HyperbolicOmegaMesh(-10, 10, 301)), [0.0, 1e-300, -1e-3, 1e3]]))
    nu = np.concatenate([g["iomega"], [1e-8, 1e4]])
    K = torch.empty((2 * len(nu), len(om)), dtype=torch.float64, device="cuda")
    i_d = torch.as_tensor(nu, device="cuda")
    o_d = torch.as_tensor(np.asarray(om), device="cuda")
    _lib.check(_lib.load().mx_iomega_kernel(i_d.data_ptr(), o_d.data_ptr(), len(nu), len(om), K.data_ptr(),
                                            ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "mx_iomega_kernel")
    ref = mb.IOmegaKernel(nu, om).fused_matrix()
    np.testing.assert_allclose(K.cpu().numpy(), ref, rtol=1e-15, atol=0)


def test_matsubara_batch_matches_reference_and_single_path(torch_cuda):
    """64 spectra of Matsubara data (g14's G as row 0) with scale_alpha = 'Ndata': row 0 passes the tiered contract
    against the real reference (which ran with scale_alpha = n_iw, not the 2 n_iw stacked rows), and every row agrees with
    the single-spectrum MaxEntLoop + IOmegaKernel run on the same row within the same contract, with identical picks."""
    g = gc.load_golden("g14_iomega_200x100.npz")
    B = 64
    G = _batch(g, B)
    j = _job(g)
    j.set_G_iw_data(g["iomega"], G)
    j.set_error(float(g["err"]))
    out = j.run()
    np.testing.assert_allclose(out.alpha, g["ref_alpha"], rtol=1e-15)
    assert out.n_sv == int(g["ref_n_sv"])
    # the kernel comes from the device fill (mx_iomega_kernel): chi2 and S get the floor gc documents for device kernels
    gc.check_against_reference(g, out.device, b=0, rtol_chi2_S=2e-7)
    om = mb.DataOmegaMesh(g["omega"])
    tolA, tolc = gc.tolerances(g, "A"), np.maximum(gc.tolerances(g, "chi2"), 2e-7)
    worst = 0.0
    for b in range(B):
        K = mb.IOmegaKernel(g["iomega"], om, beta=float(g["beta"]))
        D = mb.FlatDefaultModel(omega=om)
        Q = mb.MaxEntCostFunction(chi2=mb.ComplexChi2(K=K, G=G[b], err=float(g["err"]) * np.ones(len(G[b]))),
                                  S=mb.NormalEntropy(D=D), H_of_v=mb.NormalH_of_v(D=D, K=K))
        ml = mb.MaxEntLoop(cost_function=Q, alpha_mesh=mb.DataAlphaMesh(g["alpha_mesh"]),
                           reduce_singular_space=float(g["reduce_singular_space"]), scale_alpha="Ndata",
                           probability="normal")
        ml.set_verbosity(mb.VerbosityFlags.Quiet)
        res = ml.run()
        np.testing.assert_allclose(res.alpha, out.alpha, rtol=1e-15)
        dA = gc.rel_A(out.A(b), res.A)
        assert np.all(dA <= tolA), (b, dA / tolA)
        dc = np.abs(out.chi2[b] / res.chi2 - 1)
        assert np.all(dc <= tolc), (b, dc / tolc)
        worst = max(worst, float(np.max(dA / tolA)), float(np.max(dc / tolc)))
        for k, name in enumerate(mb.batched.ANALYZER_NAMES[:4]):
            assert int(out.alpha_index[b, k]) == int(res.analyzer_results[name]["alpha_index"]), (b, name)
    print("worst deviation / tolerance over the 64 rows: %.3g" % worst)


def test_matsubara_error_models_in_one_launch(torch_cuda):
    """[B] and [B, n_iw] errors of Matsubara data in one launch equal separate launches of each error model (an error
    per Matsubara point is repeated for the Re and Im rows)."""
    g = gc.load_golden("g14_iomega_200x100.npz")
    B, n_iw = 6, len(g["iomega"])
    G = _batch(g, B, seed=5)
    err = float(g["err"])
    tolA = gc.tolerances(g, "A")

    def check(out, b, ref, what):
        dA = gc.rel_A(out.A(b), ref.A(0))
        assert np.all(dA <= tolA), (what, b, dA / tolA)
        np.testing.assert_allclose(out.chi2[b], ref.chi2[0], rtol=1e-7, err_msg="%s %d" % (what, b))
        assert np.array_equal(out.alpha_index[b, :4], ref.alpha_index[0, :4]), (what, b)

    def single(Gb, e):
        j = _job(g)
        j.set_G_iw_data(g["iomega"], Gb[None, :])
        j.set_error(e)
        return j.run()

    sig = err * np.array([1.0, 2.0, 0.5, 1.0, 3.0, 0.7])
    j = _job(g)
    j.set_G_iw_data(g["iomega"], G)
    j.set_error(sig)
    out = j.run()
    for b in range(B):
        check(out, b, single(G[b], sig[b]), "sigma")
    rng = np.random.RandomState(3)
    vecs = err * (1.0 + 0.5 * rng.rand(3, n_iw))
    which = np.array([0, 1, 2, 1, 0, 2])
    j = _job(g)
    j.set_G_iw_data(g["iomega"], G)
    j.set_error(vecs[which])
    out = j.run()
    assert j._error_plan(B)[0] == "groups"
    for b in range(B):
        check(out, b, single(G[b], vecs[which[b]]), "vector")


def test_matsubara_threshold_skip_uses_the_modulus(torch_cuda):
    """An all-zero row is skipped; a row whose real and imaginary parts are both below G_threshold but whose modulus
    is not is continued (MaxEntLoop.run takes max |G(i omega_n)|); the other rows are unchanged by a bit."""
    from maxent_b200 import _lib
    g = gc.load_golden("g14_iomega_200x100.npz")
    G = _batch(g, 5)
    thr = 1e-10
    G[1] = 0.0
    G[3] = 0.0
    G[3, 7] = 0.8 * thr * (1 + 1j)                 # |G| = 1.13 thr: continued
    G[4] = 0.0
    G[4, 7] = 0.6 * thr * (1 + 1j)                 # |G| = 0.85 thr: skipped
    j = _job(g, G_threshold=thr)
    j.set_G_iw_data(g["iomega"], G)
    j.set_error(float(g["err"]))
    out = j.run()
    assert out.zero_elements == [1, 4]
    assert bool((out.device.status[[1, 4]] == _lib.STATUS_SKIPPED).all()) and np.all(out.alpha_index[[1, 4]] == -1)
    assert np.all(np.isfinite(out.chi2[3]))
    j2 = _job(g, G_threshold=thr)
    j2.set_G_iw_data(g["iomega"], G[[0, 2, 3]])
    j2.set_error(float(g["err"]))
    ref = j2.run()
    np.testing.assert_array_equal(out.chi2[[0, 2, 3]], ref.chi2)
    np.testing.assert_array_equal(out.A_out[[0, 2, 3]], ref.A_out)


def test_matsubara_covariance_raises(torch_cuda):
    g = gc.load_golden("g14_iomega_200x100.npz")
    j = _job(g)
    j.set_G_iw_data(g["iomega"], _batch(g, 2))
    with pytest.raises(NotImplementedError):
        j.set_cov(np.eye(2 * len(g["iomega"])))
