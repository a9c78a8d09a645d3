"""Whitening groups of BatchedTauMaxEnt across runs that leave spectra below G_threshold out of the launch: a spectrum's
group, and the SharedProblem it runs with, do not depend on which other spectra of the batch are live."""
import numpy as np
import pytest

import maxent_b200 as mb
from maxent_b200 import batched
from oracle import maxent_oracle as mo

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("model", ["err", "cov"])
def test_groups_are_kept_across_a_run_with_skipped_spectra(model):
    """One error vector (err[B, n_tau]) or covariance (cov[B, n, n]) per spectrum, three distinct ones, and spectrum 0 is
    the only spectrum of its group.  The same job runs once with spectrum 0 below G_threshold and once with every
    spectrum live: each run is bitwise the run of a fresh job on the same batch."""
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    n_tau = 120
    pr = mo.synthetic_problem(n_tau, 60, beta=20.0, mu=[0.5, -0.5, 1.0, 0.0], sigma=1e-3, seed=3)
    mesh = mo.log_alpha_mesh(0.5, 500.0, 8)
    rng = np.random.RandomState(8)
    which = np.array([0, 1, 2, 1])
    if model == "err":
        # np.unique numbers the groups in sorted order: spectrum 0's vector sorts first
        vecs = 1e-3 * np.array([0.5, 1.0, 1.5])[:, None] * (1.0 + 0.2 * rng.rand(3, n_tau))
        errors = vecs[which]
    else:
        # groups of covariances are numbered in the order of first appearance: spectrum 0's comes first
        i = np.arange(n_tau)
        C = 1e-6 * (np.eye(n_tau) + 0.4 * np.exp(-np.abs(i[:, None] - i[None, :]) / 2.5))
        errors = np.stack([c * C for c in (0.5, 1.0, 1.5)])[which]

    def job():
        j = batched.BatchedTauMaxEnt(reduce_singular_space=1e-10)
        j.set_kernel_tau(pr["tau"], batched.DataOmegaMesh(pr["omega"]), beta=20.0)
        j.alpha_mesh = mb.DataAlphaMesh(mesh)
        if model == "err":
            j.set_error(errors)
        else:
            j.set_cov(errors)
        return j

    def assert_same(out, ref, what):
        assert out.zero_elements == ref.zero_elements, what
        for name in ("chi2", "S", "Q", "probability", "n_iter", "converged", "alpha_index", "A_out"):
            np.testing.assert_array_equal(getattr(out, name), getattr(ref, name), err_msg="%s %s" % (what, name))
        assert torch.equal(out.device.A, ref.device.A), what

    G = np.array(pr["G"][:4])
    G_skip = G.copy()
    G_skip[0] = 0.0
    j = job()
    first = j.run(G_skip)
    assert first.zero_elements == [0]
    assert_same(first, job().run(G_skip), "spectrum 0 skipped")
    again = j.run(G)
    assert again.zero_elements == []
    assert_same(again, job().run(G), "every spectrum live")
