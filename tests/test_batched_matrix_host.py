"""Host-side logic of the batched matrix front ends (maxent_b200/batched_matrix.py): the element plan of the two passes,
the assembly of the result arrays from pass outputs, and input validation.  No device needed."""
import numpy as np
import pytest

import maxent_b200 as mb
from maxent_b200 import _lib
from maxent_b200.batched_matrix import element_plan, BatchedMatrixMaxEntResult


@pytest.mark.parametrize("herm", [True, False])
@pytest.mark.parametrize("cplx", [True, False])
def test_element_plan(herm, cplx):
    B, M = 3, 3
    diag, off = element_plan(B, M, use_hermiticity=herm, use_complex=cplx)
    assert diag.tolist() == [[b, i, i, 0] for b in range(B) for i in range(M)]
    parts = [0, 1] if cplx else [0]
    want = [[b, i, j, c] for b in range(B) for i in range(M) for j in range(M) if i != j and (i < j or not herm)
            for c in parts]
    assert off.tolist() == want
    assert len(off) == B * (M * (M - 1) // (2 if herm else 1)) * len(parts)


def _job(cplx, herm, B=2, M=2, n_tau=6):
    job = mb.BatchedPoormanMaxEnt(use_hermiticity=herm, use_complex=cplx)
    job.set_G_tau_data(np.linspace(0, 1, n_tau), np.ones((B, M, M, n_tau)))
    job.omega = mb.HyperbolicOmegaMesh(-1, 1, 4)
    return job


def _synthetic_pass(plan, n_alpha, n_omega, tag):
    """Pass output whose every entry encodes (row, tag): value = 100 * tag + row."""
    R = len(plan)
    val = (100.0 * tag + np.arange(R))
    return dict(chi2=np.repeat(val[:, None], n_alpha, 1), S=np.repeat(val[:, None], n_alpha, 1),
                Q=np.repeat(val[:, None], n_alpha, 1), logp=np.full((R, n_alpha), np.nan),
                n_iter=np.ones((R, n_alpha), dtype=np.int32),
                status=np.full((R, n_alpha), _lib.STATUS_CONVERGED, dtype=np.int32),
                alpha_index=np.repeat(np.arange(R, dtype=np.int32)[:, None], _lib.N_ANALYZERS, 1),
                A_out=np.repeat(val[:, None, None], _lib.N_ANALYZERS, 1).repeat(n_omega, 2),
                zero=np.zeros(R, dtype=bool), bad=np.zeros(R, dtype=bool))


@pytest.mark.parametrize("herm", [True, False])
@pytest.mark.parametrize("cplx", [True, False])
def test_result_assembly_hermiticity(herm, cplx):
    B, M, n_alpha, n_omega = 2, 2, 3, 4
    job = _job(cplx, herm, B, M)
    plans = element_plan(B, M, herm, cplx)
    host = [_synthetic_pass(plans[0], n_alpha, n_omega, 1), _synthetic_pass(plans[1], n_alpha, n_omega, 2)]
    host[1]["zero"][:] = False
    out = BatchedMatrixMaxEntResult()
    out.matrix_structure, out.use_hermiticity, out.complex_elements = (M, M), herm, cplx
    out.alpha, out._shape = np.ones(n_alpha), (M, M) + ((2,) if cplx else ())
    job._fill(out, plans, host, B, M)
    assert out.A_out.shape == (B, M, M, _lib.N_ANALYZERS, n_omega)
    assert out.chi2.shape == (B,) + out._shape + (n_alpha,)
    assert out.alpha_index.shape == (B,) + out._shape + (_lib.N_ANALYZERS,)
    for b in range(B):
        for i in range(M):
            assert np.all(out.A_out[b, i, i].real == 100 + b * M + i)
            if cplx:
                assert np.all(out.A_out[b, i, i].imag == 0) and (i, i, 1) in out.zero_elements[b]
        off = [tuple(r) for r in plans[1]]
        re = off.index((b, 0, 1, 0))
        assert np.all(out.A_out[b, 0, 1].real == 200 + re)
        if cplx:
            assert np.all(out.A_out[b, 0, 1].imag == 200 + re + 1)
        if herm:
            # (1, 0) was not continued: A_out is the conjugate of (0, 1), the scalars stay NaN
            np.testing.assert_array_equal(out.A_out[b, 1, 0], np.conj(out.A_out[b, 0, 1]))
            assert np.all(np.isnan(out.chi2[b, 1, 0])) and np.all(out.alpha_index[b, 1, 0] == -1)
        else:
            assert np.all(out.A_out[b, 1, 0].real == 200 + off.index((b, 1, 0, 0)))


def test_result_assembly_skips():
    """A below-threshold element is listed in zero_elements with A_out = 0; a Poorman element without default model is
    listed in skipped_elements with A_out = NaN; neither is copied by hermiticity from a missing source."""
    B, M = 2, 2
    job = _job(False, True, B, M)
    plans = element_plan(B, M, True, False)
    host = [_synthetic_pass(plans[0], 3, 4, 1), _synthetic_pass(plans[1], 3, 4, 2)]
    host[0]["zero"][3] = True                   # (b=1, 1, 1)
    host[1]["bad"][1] = True                    # (b=1, 0, 1)
    out = BatchedMatrixMaxEntResult()
    out.matrix_structure, out.use_hermiticity, out.complex_elements = (M, M), True, False
    out.alpha, out._shape = np.ones(3), (M, M)
    job._fill(out, plans, host, B, M)
    assert out.zero_elements == [[], [(1, 1)]] and out.skipped_elements == [[], [(0, 1)]]
    assert np.all(out.A_out[1, 1, 1] == 0) and np.all(np.isnan(out.chi2[1, 1, 1]))
    assert np.all(np.isnan(out.A_out[1, 0, 1])) and np.all(np.isnan(out.A_out[1, 1, 0]))
    assert np.all(out.A_out[0, 1, 0] == out.A_out[0, 0, 1])


def test_error_shapes():
    B, M, n_tau = 3, 2, 6
    job = _job(False, True, B, M, n_tau)
    kinds = {(): "shared", (n_tau,): "shared", (M, M, n_tau): "element", (B, M, M): "spectrum"}
    for shape, kind in kinds.items():
        job.set_error(np.full(shape, 1e-3) if shape else 1e-3)
        assert job._error_kind(B, M) == kind
    job.set_error(np.ones((M, M, n_tau - 1)))
    with pytest.raises(ValueError):
        job._error_kind(B, M)
    job.set_error(np.ones((B, M, M + 1)))
    with pytest.raises(ValueError):
        job._error_kind(B, M)
    job.set_cov(np.eye(n_tau))
    assert job._error_kind(B, M) == "cov"
    with pytest.raises(NotImplementedError):
        job.set_cov(np.ones((M, M, n_tau, n_tau)))
    with pytest.raises(NotImplementedError):
        job.set_preblur(0.1)
    with pytest.raises(ValueError):
        job.set_G_tau_data(np.linspace(0, 1, n_tau), np.ones((B, M, M + 1, n_tau)))
    with pytest.raises(ValueError):
        mb.BatchedPoormanMaxEnt(analyzer_offdiag_D="NoSuchAnalyzer")


def test_error_groups_by_element():
    """Per-element error vectors become one whitening group per element, indexed by element (no per-row copies)."""
    B, M, n_tau = 2, 2, 6
    job = _job(False, False, B, M, n_tau)
    err = np.arange(1, M * M * n_tau + 1, dtype=float).reshape(M, M, n_tau)
    job.set_error(err)
    diag, off = element_plan(B, M, False, False)
    job._put_error(job.maxent_offdiagonal, "element", off)
    mode, index, specs = job.maxent_offdiagonal._error_plan(len(off))
    assert mode == "groups" and len(specs) == 2
    for r, (b, i, j, c) in enumerate(off):
        np.testing.assert_array_equal(specs[index[r]][1], err[i, j])
    job._put_error(job.maxent_diagonal, "element", diag)
    mode, index, specs = job.maxent_diagonal._error_plan(len(diag))
    assert [specs[index[r]][1][0] for r in range(len(diag))] == [err[i, i, 0] for b in range(B) for i in range(M)]


def test_namespace():
    for name in ("BatchedElementwiseMaxEnt", "BatchedPoormanMaxEnt", "BatchedMatrixMaxEntResult"):
        assert hasattr(mb, name)
    assert issubclass(mb.BatchedPoormanMaxEnt, mb.BatchedElementwiseMaxEnt)
    from maxent_b200 import ops
    assert "poorman_models" in ops.OPERATORS


def _dropin_A_out(host, plans, b, M, herm, cplx, zero_elements, n_omega):
    """A_out of matrix b as MaxEntResult.get_A_out assembles it from the same analyzer outputs, per analyzer slot."""
    from maxent_b200.maxent_result import MaxEntResult
    res = MaxEntResult(matrix_structure=(M, M), complex_elements=cplx, use_hermiticity=herm)
    res.add_sweep(dict(alpha=np.ones(3), omega=np.arange(n_omega)), matrix_element=(0, 0), complex_index=0)
    for plan, got in zip(plans, host):
        for r, (bb, i, j, c) in enumerate(plan):
            if bb != b or got["zero"][r] or got["bad"][r]:
                continue
            slot = res._get_element(res._results_from_analyzers, (i, j, c) if cplx else (i, j))
            for k, name in enumerate(mb.batched.ANALYZER_NAMES):
                slot[name] = dict(A_out=got["A_out"][r, k])
    res._zero_elements = list(zero_elements)
    return np.stack([res.get_A_out(name) for name in mb.batched.ANALYZER_NAMES], axis=-2)


@pytest.mark.parametrize("herm", [True, False])
@pytest.mark.parametrize("which", ["re", "im", "both", "none"])
def test_result_assembly_matches_get_A_out(herm, which):
    """A complex off-diagonal with one part below G_threshold keeps its computed part: the batched A_out equals what
    MaxEntResult.get_A_out assembles from the same per-part outputs (zeros first, then computed parts, then the
    hermiticity copies of computed parts)."""
    B, M, n_omega = 2, 2, 4
    job = _job(True, herm, B, M)
    plans = element_plan(B, M, herm, True)
    host = [_synthetic_pass(plans[0], 3, n_omega, 1), _synthetic_pass(plans[1], 3, n_omega, 2)]
    off = [tuple(r) for r in plans[1]]
    for c in {"re": [0], "im": [1], "both": [0, 1], "none": []}[which]:
        host[1]["zero"][off.index((1, 0, 1, c))] = True
    out = BatchedMatrixMaxEntResult()
    out.matrix_structure, out.use_hermiticity, out.complex_elements = (M, M), herm, True
    out.alpha, out._shape = np.ones(3), (M, M, 2)
    job._fill(out, plans, host, B, M)
    for b in range(B):
        want = _dropin_A_out(host, plans, b, M, herm, True, out.zero_elements[b], n_omega)
        np.testing.assert_array_equal(out.A_out[b], want)
        assert all(type(x) is int for el in out.zero_elements[b] for x in el)
    if which == "im":
        k = off.index((1, 0, 1, 0))
        assert np.all(out.A_out[1, 0, 1].real == 200 + k) and np.all(out.A_out[1, 0, 1].imag == 0)
        assert np.all(out.chi2[1, 0, 1, 0] == 200 + k)
