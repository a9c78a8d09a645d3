"""GPU tests of the batched matrix front ends (BatchedElementwiseMaxEnt, BatchedPoormanMaxEnt): runs of the real
reference (tests/golden), the drop-in classes per matrix, batch-composition independence (bitwise), the device default
models of mx_poorman_models, per-element / per-spectrum error models and skips."""
import numpy as np
import pytest

import maxent_b200 as mb
from tests import gpu_common as gc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _cuda():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"


def _batched(cls, g, G, err=None, **kw):
    job = cls(**kw)
    job.set_G_tau_data(g["tau"], G)
    job.omega = mb.DataOmegaMesh(g["omega"])
    job.alpha_mesh = mb.DataAlphaMesh(g["alpha_mesh"])
    job.set_error(float(g["err"]) if err is None else err)
    return job


def _dropin(cls, tau, G, omega, alpha_mesh, err, **kw):
    ew = cls(**kw)
    ew.set_verbosity(mb.VerbosityFlags.Quiet)
    ew.set_G_tau_data(tau, G)
    ew.omega = omega
    ew.alpha_mesh = alpha_mesh
    ew.set_error(err)
    return ew.run()


def _other(G):
    """A different matrix of the same kind: diagonal swapped, off-diagonal conjugated and scaled."""
    H = np.array(G)
    H[0, 0], H[1, 1] = G[1, 1], G[0, 0]
    H[0, 1], H[1, 0] = 0.7 * np.conj(G[0, 1]), 0.7 * np.conj(G[1, 0])
    return H


def _same(a, b):
    np.testing.assert_array_equal(np.asarray(a), np.asarray(b))


def _assert_matrix_equal(out1, b1, out2, b2):
    for name in ("A_out", "chi2", "S", "Q", "alpha_index", "n_iter", "converged"):
        _same(getattr(out1, name)[b1], getattr(out2, name)[b2])
    _same(out1.A(b1), out2.A(b2))


@pytest.fixture(scope="module")
def g10_batch():
    g = gc.load_golden("g10_poorman_2x2.npz")
    G = np.stack([g["G"], _other(g["G"]), g["G"]])
    return g, G, _batched(mb.BatchedPoormanMaxEnt, g, G, use_hermiticity=False).run()


def test_poorman_matches_reference_run(g10_batch):
    g, G, out = g10_batch
    for b in (0, 2):
        gc.check_matrix_result(out.result(b), g)
    assert out[1].matrix_structure == (2, 2) and out[-1].zero_elements == []


def test_complex_poorman_matches_reference_run():
    g = gc.load_golden("g12_complex_poorman_2x2.npz")
    G = np.stack([g["G"], _other(g["G"]), g["G"]])
    out = _batched(mb.BatchedPoormanMaxEnt, g, G, use_hermiticity=True, use_complex=True).run()
    assert np.iscomplexobj(out.A_out) and out.A_out.shape[:3] == (3, 2, 2)
    for b in (0, 2):
        res = out.result(b)
        gc.check_matrix_result(res, g)
        A_out = res.A_out
        for iw in range(A_out.shape[-1]):
            assert np.all(A_out[..., iw] == A_out[..., iw].conjugate().transpose())
        for iw in range(out.A_out.shape[-1]):
            X = out.A_out[b, :, :, 0, iw]
            assert np.all(X == X.conjugate().T)


@pytest.mark.parametrize("name,herm,cplx", [("g6_elementwise_2x2.npz", True, False),
                                            ("g11_complex_elementwise_2x2.npz", False, True)])
def test_elementwise_matches_reference_run(name, herm, cplx):
    g = gc.load_golden(name)
    G = np.stack([g["G"], _other(g["G"]), g["G"]])
    out = _batched(mb.BatchedElementwiseMaxEnt, g, G, use_hermiticity=herm, use_complex=cplx).run()
    for b in (0, 2):
        gc.check_matrix_result(out.result(b), g)
    _assert_matrix_equal(out, 0, out, 2)


def test_batch_composition_independence(g10_batch):
    """Matrix results do not depend on which other matrices share the batch or where they sit: both passes and the
    device default models, bitwise."""
    g, G, out = g10_batch
    _assert_matrix_equal(out, 0, out, 2)
    alone = _batched(mb.BatchedPoormanMaxEnt, g, G[:1], use_hermiticity=False).run()
    _assert_matrix_equal(out, 0, alone, 0)
    rev = _batched(mb.BatchedPoormanMaxEnt, g, np.stack([G[1], G[0], _other(G[1])]), use_hermiticity=False).run()
    _assert_matrix_equal(out, 0, rev, 1)
    _assert_matrix_equal(out, 1, rev, 0)


def test_device_default_models(g10_batch):
    """mx_poorman_models: D bit for bit as numpy forms it, v0 = V'^T log(arg) to 1e-13, ok = 0 exactly where a diagonal
    partner holds NaN."""
    g, G, _ = g10_batch
    job = _batched(mb.BatchedPoormanMaxEnt, g, G, use_hermiticity=False)
    plans, (r1, _), _, _ = job.run_device(diagonal_only=True)
    B, M = G.shape[:2]
    _, off = mb.batched_matrix.element_plan(B, M, False, False)
    rows = np.stack([off[:, 0] * M + off[:, 1], off[:, 0] * M + off[:, 2]], axis=1)
    A_out = r1.A_out.clone()
    D, v0, ok = job.default_models(A_out, off)
    A = A_out[:, 0].cpu().numpy()
    prob = job.maxent_offdiagonal.prepare()
    delta = prob.delta.cpu().numpy()
    n_om = len(delta)
    D_np = (np.sqrt(A[rows[:, 0]] * A[rows[:, 1]]) + 1e-6) * delta
    _same(D.cpu().numpy()[:, :n_om], D_np)
    assert np.all(D.cpu().numpy()[:, n_om:] == 0)
    H0 = D_np * delta
    arg = (H0 + np.sqrt(H0 ** 2 + 4 * D_np ** 2)) / (2 * D_np)
    v_np = np.log(np.where(np.abs(arg) <= 1e-100, 1e-100, arg)) @ prob.Vp.cpu().numpy()
    assert np.max(np.abs(v0.cpu().numpy() - v_np)) <= 1e-13 * np.max(np.abs(v_np))
    assert np.all(ok.cpu().numpy() == 1)
    A_out[3, 0, 5] = float("nan")                                # diagonal (b=1, i=1)
    _, _, ok = job.default_models(A_out, off)
    want = ~((rows[:, 0] == 3) | (rows[:, 1] == 3))
    _same(ok.cpu().numpy(), want.astype(np.int32))
    with pytest.raises(ValueError):
        job.default_models(A_out, off + np.array([10, 0, 0, 0]))


def _tiered(A, chi2, base, floor):
    """A and chi2 within 1e-8 where the single run reproduces itself, 10x its noise floor elsewhere."""
    nA, nc = floor
    tolA = np.maximum(gc.RTOL_WELL_DETERMINED, gc.NOISE_FACTOR * nA)
    tolc = np.maximum(gc.RTOL_WELL_DETERMINED, gc.NOISE_FACTOR * nc)
    dA = gc.rel_A(A, base["A"])
    assert np.all(dA <= tolA), dA / tolA
    dc = np.abs(chi2 / base["chi2"] - 1)
    assert np.all(dc <= tolc), dc / tolc


def _element_floor(run, base_res, elements):
    """Per element, the noise floor of a drop-in run under the gc.EPS perturbations of its data."""
    floors = {}
    runs = [run(1.0 + e) for e in gc.EPS]
    for el in elements:
        nA, nc = np.zeros(len(base_res.alpha)), np.zeros(len(base_res.alpha))
        for r in runs:
            nA = np.maximum(nA, gc.rel_A(r.A[el], base_res.A[el]))
            nc = np.maximum(nc, np.abs(r.chi2[el] / base_res.chi2[el] - 1))
        floors[el] = (gc.running_max(nA), gc.running_max(nc))
    return floors


def test_against_dropin_at_realistic_shape():
    """16 random complex Hermitian 2x2 matrices at n_tau 1000, n_omega 400, 60 alphas; four of them against
    PoormanMaxEnt run per matrix: identical LineFit / Chi2Curvature picks, A and chi2 under the tiered rule."""
    tau, omega, G = mb.batched_matrix.synthetic_matrix_batch(1000, 400, 16, seed=11)
    alpha = mb.LogAlphaMesh(1e-4, 1e3, 60)
    job = mb.BatchedPoormanMaxEnt(use_hermiticity=True, use_complex=True)
    job.set_G_tau_data(tau, G)
    job.omega, job.alpha_mesh = omega, alpha
    job.set_error(1e-4)
    out = job.run()
    elements = [(0, 0, 0), (1, 1, 0), (0, 1, 0), (0, 1, 1)]
    for b in (0, 5, 10, 15):
        def run(f, b=b):
            return _dropin(mb.PoormanMaxEnt, tau, G[b] * f, omega, alpha, 1e-4, use_hermiticity=True, use_complex=True)
        ref = run(1.0)
        floors = _element_floor(run, ref, elements)
        res = out.result(b)
        for el in elements:
            for an in ("LineFitAnalyzer", "Chi2CurvatureAnalyzer"):
                assert (res.analyzer_results[el[0]][el[1]][el[2]][an]["alpha_index"]
                        == ref.analyzer_results[el[0]][el[1]][el[2]][an]["alpha_index"]), (b, el, an)
            _tiered(res.A[el], res.chi2[el], dict(A=ref.A[el], chi2=ref.chi2[el]), floors[el])


def _single_plusminus(g, Gij, err, D, f=1.0):
    tm = mb.TauMaxEnt(cost_function="plusminus")
    tm.set_verbosity(mb.VerbosityFlags.Quiet)
    tm.set_G_tau_data(g["tau"], Gij * f)
    tm.omega = mb.DataOmegaMesh(g["omega"])
    tm.alpha_mesh = mb.DataAlphaMesh(g["alpha_mesh"])
    tm.D = mb.DataDefaultModel(D, tm.omega)
    tm.set_error(err)
    return tm.run()


@pytest.mark.parametrize("kind", ["element", "spectrum"])
def test_error_models_per_element_and_per_spectrum(kind):
    """Every off-diagonal element agrees with one TauMaxEnt(cost_function='plusminus') run carrying that element's error
    and its Poorman default model."""
    g = gc.load_golden("g10_poorman_2x2.npz")
    G = np.stack([g["G"], _other(g["G"])])
    B, M, n_tau = 2, 2, len(g["tau"])
    e0 = float(g["err"])
    if kind == "element":
        err = e0 * (1.0 + 0.25 * np.arange(M * M)[:, None] / (M * M) + 0.1 * np.linspace(0, 1, n_tau)[None, :])
        err = err.reshape(M, M, n_tau)
    else:
        err = e0 * (1.0 + 0.2 * np.arange(B * M * M).reshape(B, M, M))
    out = _batched(mb.BatchedPoormanMaxEnt, g, G, err=err, use_hermiticity=False).run()
    for b in range(B):
        res = out.result(b)
        for (i, j) in ((0, 1), (1, 0)):
            e = err[i, j] if kind == "element" else float(err[b, i, j])
            D = np.sqrt(res.analyzer_results[i][i]["LineFitAnalyzer"]["A_out"]
                        * res.analyzer_results[j][j]["LineFitAnalyzer"]["A_out"]) + 1e-6
            ref = _single_plusminus(g, G[b, i, j], e, D)
            runs = [_single_plusminus(g, G[b, i, j], e, D, 1.0 + x) for x in gc.EPS]
            nA = gc.running_max(np.max([gc.rel_A(r.A, ref.A) for r in runs], axis=0))
            nc = gc.running_max(np.max([np.abs(r.chi2 / ref.chi2 - 1) for r in runs], axis=0))
            _tiered(res.A[i, j], res.chi2[i, j], dict(A=ref.A, chi2=ref.chi2), (nA, nc))
            assert (res.analyzer_results[i][j]["LineFitAnalyzer"]["alpha_index"]
                    == ref.analyzer_results["LineFitAnalyzer"]["alpha_index"])


def test_per_spectrum_models_with_error_groups():
    """BatchedTauMaxEnt.run(G, D=...) with one error vector per spectrum (default models and whitening groups in one
    launch) agrees with one run per group."""
    g = gc.load_golden("g10_poorman_2x2.npz")
    n_tau = len(g["tau"])
    G = np.stack([g["G"][0, 1], 0.8 * g["G"][0, 1], g["G"][1, 0], 1.1 * g["G"][0, 1]])
    om = mb.DataOmegaMesh(g["omega"])
    w = np.asarray(om)
    D = np.stack([np.exp(-w ** 2 / s) / np.sqrt(np.pi * s) + 1e-6 for s in (1.0, 2.0, 3.0, 4.0)]) * om.delta
    e0 = float(g["err"])
    errs = np.stack([e0 * np.ones(n_tau), e0 * (1 + 0.3 * np.linspace(0, 1, n_tau))])
    index = np.array([0, 1, 1, 0])

    def job(err):
        t = mb.BatchedTauMaxEnt(cost_function="plusminus")
        t.set_G_tau_data(g["tau"], G)
        t.omega, t.alpha_mesh = om, mb.DataAlphaMesh(g["alpha_mesh"])
        t.set_error(err)
        return t
    out = job(errs[index]).run(G, D=D)
    for grp in range(2):
        sel = np.nonzero(index == grp)[0]
        ref = job(errs[grp]).run(G[sel], D=D[sel])
        _same(out.alpha_index[sel], ref.alpha_index)
        for k, b in enumerate(sel):
            A, Ar = out.A(b), ref.A(k)
            n = ref.alpha_index[k, 0] + 1                    # up to the LineFit pick: the well-determined range
            assert np.max(gc.rel_A(A, Ar)[:n]) <= 1e-7
            np.testing.assert_allclose(out.chi2[b, :n], ref.chi2[k, :n], rtol=1e-7)


def test_skips(g10_batch):
    """A zero diagonal element is in zero_elements; the off-diagonals that need it are not continued (NaN, listed in
    skipped_elements); the other matrices are bitwise those of a run without that matrix."""
    g, G, out = g10_batch
    Z = np.array(G[1])
    Z[1, 1] = 0.0
    Gz = np.stack([G[0], Z, G[2]])
    outz = _batched(mb.BatchedPoormanMaxEnt, g, Gz, use_hermiticity=False).run()
    assert outz.zero_elements[1] == [(1, 1)] and sorted(outz.skipped_elements[1]) == [(0, 1), (1, 0)]
    assert outz.zero_elements[0] == [] and outz.skipped_elements[0] == []
    assert np.all(outz.A_out[1, 1, 1] == 0)
    assert np.all(np.isnan(outz.A_out[1, 0, 1])) and np.all(np.isnan(outz.chi2[1, 1, 0]))
    res = outz.result(1)
    assert res.zero_elements == [(1, 1)] and sorted(res.skipped_elements) == [(0, 1), (1, 0)]
    without = _batched(mb.BatchedPoormanMaxEnt, g, Gz[[0, 2]], use_hermiticity=False).run()
    _assert_matrix_equal(outz, 0, without, 0)
    _assert_matrix_equal(outz, 2, without, 1)
