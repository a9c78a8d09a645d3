"""The fused alpha sweep at the edge shapes of its V' stream, against the oracle and against itself.

V' streams in chunks of CH = 8 k-tiles (64 omega rows): nch = ceil(n_kt / 8) chunks, the last one holding
n_kt - 8 (nch - 1) tiles.  The narrow instantiations (NT <= 10 tiles) stage the chunks in a ring of NST buffers whose
mbarrier phases are counted across every pass and every spectrum a persistent CTA takes (Ctl.gchunk); the wide ones
(NT >= 12) read V' from L2, the T-pass striding k-tiles by NWARP = 8 and the H-pass prefetching one k-tile ahead.  In
a partial last chunk the warps past the last tile see stale staging memory, kept out of y, S and Z only by the guards
of the T-pass and H-pass.  The case table below puts every narrow NT on meshes of one chunk (n_omega = n_sv, a
partial chunk), on two and three chunks whose last holds one tile, and on a long mesh whose last chunk holds seven;
the three-stage ring (NT = 9, 10) on two to five chunks, each with a partial last chunk, where the steady-state refill
runs from three on; the wide instantiations at n_omega = n_sv, at n_kt = 1 (mod 8) and on both sides of 2 NWARP.

Each case is held to the tiered oracle contract (A and chi2 within 1e-8 where the oracle reproduces itself, 10x its
measured floor elsewhere) and to two checks the oracle cannot make, since it does not see the chunk geometry: chi2 and
S recomputed in float64 from the returned A with the full kernel, and stationarity at the converged alphas.  Several
spectra per CTA must each give the bits of their run alone; one alpha must match the oracle and give the analyzers'
one-point results.  test_case_table_geometry (no GPU) checks the table itself.
"""
import collections
import ctypes

import numpy as np
import pytest

from oracle import maxent_oracle as mo
from tests import gpu_common as gc

CH = 8                      # k-tiles per staged chunk (mx_sweep2.cuh: CH = NWARP)
NWARP = 8
# Stages of the V' ring per tile count: Lay<NT>::NST = stage_count(NT) in maxent_b200/csrc/mx_sweep2.cuh.  The wide
# instantiations (NT >= 12) have no ring (0).  A change of stage_count() makes this table stale, not the coverage lost.
NST = {4: 2, 5: 2, 6: 2, 7: 2, 8: 2, 9: 3, 10: 3, 12: 0, 16: 0, 32: 0}
ERR = 1e-4
CUT = 1e-9

Case = collections.namedtuple("Case", "nt nst n_sv n_om nch last variants model")


def _case(nt, nst, n_sv, n_om, nch, last, pm=False, model=False):
    return Case(nt, nst, n_sv, n_om, nch, last, ("normal", "plusminus") if pm else ("normal",), model)


# (NT, NST, n_sv, n_omega, nch, last-chunk tiles): the geometry each row claims, checked by test_case_table_geometry.
# pm: the plus-minus cost function as well (the one-tile-last-chunk row of every narrow NT, one wide shape);
# model: a default model per spectrum, D[B, n_omega] at odd n_omega (half the narrow rows).
CASES = [
    # narrow, two stages
    _case(4, 2, 21, 21, 1, 3, model=True),            # n_omega = n_sv
    _case(4, 2, 21, 41, 1, 6),                        # partial chunk, 8k + 1 rows
    _case(4, 2, 21, 65, 2, 1, pm=True, model=True),
    _case(4, 2, 21, 129, 3, 1),
    _case(4, 2, 21, 1009, 16, 7, model=True),
    _case(5, 2, 35, 35, 1, 5),
    _case(5, 2, 35, 49, 1, 7, model=True),
    _case(5, 2, 35, 67, 2, 1, pm=True),
    _case(5, 2, 35, 131, 3, 1, model=True),
    _case(5, 2, 35, 1011, 16, 7),
    _case(6, 2, 43, 43, 1, 6, model=True),
    _case(6, 2, 43, 49, 1, 7),
    _case(6, 2, 43, 69, 2, 1, pm=True, model=True),
    _case(6, 2, 43, 133, 3, 1),
    _case(6, 2, 43, 1013, 16, 7, model=True),
    _case(7, 2, 49, 49, 1, 7),                        # n_omega = n_sv = 8k + 1
    _case(7, 2, 49, 71, 2, 1, pm=True, model=True),
    _case(7, 2, 49, 135, 3, 1),
    _case(7, 2, 49, 1015, 16, 7, model=True),
    _case(8, 2, 57, 57, 1, 8),                        # n_omega = n_sv: one full chunk (no partial chunk at n_sv >= 57)
    _case(8, 2, 57, 72, 2, 1, pm=True),
    _case(8, 2, 57, 135, 3, 1, model=True),
    _case(8, 2, 57, 1016, 16, 7),
    # narrow, three stages: the refill runs from nch = 3 on
    _case(9, 3, 69, 69, 2, 1, pm=True, model=True),   # n_omega = n_sv
    _case(9, 3, 69, 147, 3, 3),
    _case(9, 3, 69, 211, 4, 3, model=True),
    _case(9, 3, 69, 285, 5, 4),
    _case(9, 3, 69, 1013, 16, 7, model=True),
    _case(10, 3, 77, 77, 2, 2),                       # n_omega = n_sv
    _case(10, 3, 77, 171, 3, 6, model=True),
    _case(10, 3, 77, 195, 4, 1, pm=True),
    _case(10, 3, 77, 299, 5, 6, model=True),
    _case(10, 3, 77, 1011, 16, 7),
    # wide: no ring; n_kt against 2 NWARP = 16
    _case(12, 0, 90, 90, 2, 4),                       # n_omega = n_sv, n_kt = 12 < 16
    _case(12, 0, 90, 131, 3, 1),                      # n_kt = 17 = 1 (mod 8), > 16
    _case(16, 0, 113, 113, 2, 7),                     # n_omega = n_sv, n_kt = 15 < 16
    _case(16, 0, 113, 131, 3, 1, pm=True),            # n_kt = 17
    _case(32, 0, 250, 250, 4, 8),                     # n_omega = n_sv, n_kt = 32 > 16
    _case(32, 0, 250, 259, 5, 1),                     # n_kt = 33 = 1 (mod 8)
]


def _name(c):
    return "nt%d-nst%d-om%d-nch%d-last%d" % (c.nt, c.nst, c.n_om, c.nch, c.last)


def _find(nt, n_om):
    return next(c for c in CASES if c.nt == nt and c.n_om == n_om)


# several spectra per CTA: one shape per NT whose nch is not a multiple of NST
MULTI = [_find(4, 129), _find(7, 135), _find(9, 211), _find(10, 299), _find(12, 131), _find(32, 259)]
# one alpha: a narrow and a wide shape
ONE_ALPHA = [_find(9, 147), _find(16, 113)]

RUNS = [(c, v) for c in CASES for v in c.variants]


def _n_tau(c):
    return c.n_om + 24                                  # kernel_problem needs n_tau >= n_omega


def _problem(c, variant, n_spectra=1):
    return gc.kernel_problem(c.n_sv, _n_tau(c), c.n_om, variant, 1000 * c.n_om + c.n_sv, n_spectra)


def _model(om):
    """A default model per spectrum (delta omega included, as DefaultModel.D): not flat, not normalised."""
    return mo.flat_default_model(om) * (1.0 + 0.5 * np.exp(-(om - 0.5) ** 2))


def _mesh(n_alpha):
    return mo.log_alpha_mesh(0.5, 500, n_alpha)


# ----------------------------------------------------------------------------------------------
# the case table (no GPU)
# ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", CASES, ids=_name)
def test_case_table_geometry(c):
    """Every row is the geometry its name claims -- NT from the sweep's tile formula, NST from the table of
    stage_count(), nch and the tiles of the last chunk from n_omega -- and its kernel keeps exactly n_sv singular values
    above the cut.  n_sv is never a multiple of 8; per-spectrum default models only at odd n_omega."""
    n_kt = (c.n_om + 7) // 8
    nch = (n_kt + CH - 1) // CH
    nt = gc.sweep_tiles(c.n_sv)
    assert (nt, NST[nt], nch, n_kt - CH * (nch - 1)) == (c.nt, c.nst, c.nch, c.last)
    assert c.n_sv % 8 != 0 and c.n_sv <= c.n_om
    assert not c.model or c.n_om % 2 == 1
    K, G, _, _ = _problem(c, "normal")
    S = np.linalg.svd(K, compute_uv=False)
    assert int(np.sum(S >= CUT)) == c.n_sv, (c, S[c.n_sv - 1:c.n_sv + 1])
    assert G.shape == (1, _n_tau(c))


def test_case_table_covers_the_stream_edges():
    """The table holds, for every narrow NT, meshes of one chunk (n_omega = n_sv among them), two and three chunks
    ending in one tile, and a long mesh ending in seven; for NT = 9, 10 two to five chunks, each with a partial last
    chunk; for every wide NT n_omega = n_sv and n_kt = 1 (mod 8), and across them n_kt below and above 2 NWARP.  The
    plus-minus cost function runs on the one-tile-last-chunk row of every narrow NT and on one wide shape, and half the
    narrow rows (give or take one) use per-spectrum default models."""
    for nt in (4, 5, 6, 7, 8):
        rows = [c for c in CASES if c.nt == nt]
        assert any(c.nch == 1 and c.n_om == c.n_sv for c in rows), nt
        assert {2, 3} <= {c.nch for c in rows if c.last == 1}, nt
        assert any(c.n_om >= 1000 and c.last == 7 for c in rows), nt
        assert any(c.last == 1 and c.nch == 2 and "plusminus" in c.variants for c in rows), nt
    for nt in (9, 10):
        rows = [c for c in CASES if c.nt == nt]
        assert {2, 3, 4, 5} <= {c.nch for c in rows if c.last < CH}, nt
        assert any(c.n_om >= 1000 for c in rows) and any(c.last == 1 and "plusminus" in c.variants for c in rows), nt
    wide = [c for c in CASES if c.nst == 0]
    for nt in (12, 16, 32):
        rows = [c for c in wide if c.nt == nt]
        assert any(c.n_om == c.n_sv for c in rows) and any((c.n_om + 7) // 8 % 8 == 1 for c in rows), nt
    n_kt = [(c.n_om + 7) // 8 for c in wide]
    assert min(n_kt) < 2 * NWARP < max(n_kt)
    assert any("plusminus" in c.variants for c in wide)
    narrow = [c for c in CASES if c.nst > 0]
    assert abs(2 * sum(c.model for c in narrow) - len(narrow)) <= 1
    assert all(c.nst == 0 or c.nch % c.nst != 0 for c in MULTI)


# ----------------------------------------------------------------------------------------------
# GPU
# ----------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "the gpu tests need a CUDA device"
    return torch


def _shared_problem(c, variant, K, om, delta):
    from maxent_b200 import engine
    prob = engine.SharedProblem(K, ERR, mo.flat_default_model(om), delta, variant=variant, reduce_singular_space=CUT)
    assert prob.n_sv == c.n_sv
    return prob


def _vs_oracle(K, G, om, D, mesh, variant, res, probability=False):
    """The tiered contract of test_all_kernel_instantiations_vs_oracle for spectrum 0 of `res`; returns the oracle run
    and the worst ratios (dA / tol, dchi2 / tol)."""
    svd = mo.kernel_svd(K, CUT)                          # the same for every perturbation of G: computed once
    kw = dict(D=D, variant=variant, reduce_singular_space=CUT, analyzers=False, svd=svd)
    o = mo.maxent_loop(K, G, ERR, om, mesh, probability=probability, **kw)
    nA, nc = gc.oracle_floor(o, lambda f: mo.maxent_loop(K, G * f, ERR, om, mesh, **kw))
    assert o["n_sv"] == res.n_sv
    tolA, tolc = np.maximum(1e-8, 10 * nA), np.maximum(1e-8, 10 * nc)
    rA = gc.rel_A(res.A[0].cpu().numpy(), o["A"]) / tolA
    rc = np.abs(res.chi2[0].cpu().numpy() / o["chi2"] - 1) / tolc
    assert np.all(rA <= 1), ("A", rA)
    assert np.all(rc <= 1), ("chi2", rc)
    return o, float(rA.max()), float(rc.max())


def _check_properties(K, G, D, delta, alpha, V, variant, res):
    """chi2 and S of spectrum 0 recomputed in float64 from the returned A with the full kernel (functions.py:358-360,
    508-510; plus-minus 544-564, 778-786), and stationarity max|dQ/dv| < 1e-4 in the kernel's singular basis V at every
    alpha (levenberg_minimizer.py:103-106), at the limits of test_full_size_properties."""
    A = res.A[0].cpu().numpy()
    H = A * delta                                        # [n_alpha, n_omega]
    r = (H @ K.T - G[None, :]) / ERR
    chi2 = np.sum(r * r, axis=1)
    assert np.all(np.abs(chi2 / res.chi2[0].cpu().numpy() - 1) < 1e-9), chi2 / res.chi2[0].cpu().numpy() - 1
    floor = np.log(1e-100)                               # safelog clamp, python/functions.py:53-56
    if variant == "normal":
        x = np.log(np.maximum(H / D, 1e-100))
        w = H
        terms = [H, -D, -H * x]
    else:
        x = np.arcsinh(H / (2 * D))                      # H = D (e^x - e^-x)
        Hp, Hm = D * np.exp(x), D * np.exp(-x)
        lp, lm = np.where(Hp / D <= 1e-100, floor, x), np.where(Hm / D <= 1e-100, floor, -x)
        w = Hp + Hm
        terms = [Hp, -D, -Hp * lp, Hm, -D, -Hm * lm]
    S = np.sum(sum(terms), axis=1)
    size = np.sum(sum(np.abs(t) for t in terms), axis=1)
    Sk = res.S[0].cpu().numpy()
    # 1e-10 relative, and the rounding of the sum itself where S cancels to near zero (large alpha: H ~ D)
    assert np.all(np.abs(S - Sk) <= 1e-10 * np.abs(Sk) + 64 * 2.0 ** -52 * size), (S, Sk)
    f = (w * ((r / ERR) @ K + alpha[:, None] * x)) @ V
    maxf = np.max(np.abs(f), axis=1)
    assert bool((res.status[0] & 1).all())
    assert np.all(maxf < 1.05e-4), maxf


def _run_case(torch, c, variant, n_alpha, probability=False):
    from maxent_b200 import engine
    K, G, om, delta = _problem(c, variant)
    prob = _shared_problem(c, variant, K, om, delta)
    D = _model(om) if c.model else None
    mesh = _mesh(n_alpha)
    alpha = mesh * _n_tau(c)
    res = engine.run_sweep(prob, G, alpha, probability=probability, D=None if D is None else D[None, :])
    torch.cuda.synchronize()
    o, wA, wc = _vs_oracle(K, G[0], om, D, mesh, variant, res, probability)
    _check_properties(K, G[0], mo.flat_default_model(om) if D is None else D, delta, alpha, prob.V.cpu().numpy(),
                      variant, res)
    return res, o, wA, wc


@pytest.mark.gpu
@pytest.mark.parametrize("c,variant", RUNS, ids=["%s-%s" % (_name(c), v) for c, v in RUNS])
def test_stream_geometry_vs_oracle(torch_cuda, c, variant):
    """One spectrum of every case against the oracle (n_alpha 5 to 7), with chi2, S and stationarity recomputed from A."""
    n_alpha = 5 + CASES.index(c) % 3
    _, _, wA, wc = _run_case(torch_cuda, c, variant, n_alpha)
    print("\nROW %s %s model=%d n_alpha=%d dA/tol=%.3g dchi2/tol=%.3g" % (_name(c), variant, c.model, n_alpha, wA, wc))


def _launch_grid(prob, alpha, B):
    """CTAs of the sweep launch for B spectra, read off the workspace the C ABI asks for: a fixed header plus the same
    number of bytes per CTA (scratch rows and, wide, the CTA's slice)."""
    from maxent_b200 import engine, ops
    p = ops.problem_struct(*engine._problem_args(prob, alpha, engine.LMParams(), 1.0))
    ws = lambda b: int(prob.lib.mx_sweep_workspace_bytes(ctypes.byref(p), b))
    per_cta = ws(2) - ws(1)
    assert per_cta > 0 and (ws(B) - ws(1)) % per_cta == 0
    return 1 + (ws(B) - ws(1)) // per_cta


@pytest.mark.gpu
@pytest.mark.parametrize("c", MULTI, ids=_name)
def test_several_spectra_per_cta(torch_cuda, c):
    """4 x (resident CTAs) + 7 spectra, three distinct ones interleaved, so that every persistent CTA takes about four
    and its chunk counter (the mbarrier parities) runs on across spectra: every output equals bit for bit the run of
    its spectrum alone (B = 1)."""
    torch = torch_cuda
    from maxent_b200 import _lib, engine
    K, G, om, delta = _problem(c, "normal", n_spectra=3)
    prob = _shared_problem(c, "normal", K, om, delta)
    alpha = torch.tensor(_mesh(6) * _n_tau(c), dtype=torch.float64, device="cuda")
    sms = int(_lib.load().mx_device_sm_count())
    resident = _launch_grid(prob, alpha, 1 << 30)
    assert sms <= resident <= 2 * sms
    B = 4 * resident + 7
    grid = _launch_grid(prob, alpha, B)
    assert grid == resident and B / grid > 4
    which = np.arange(B) % 3
    res = engine.run_sweep(prob, G[which], alpha)
    fields = ("A", "chi2", "S", "Q", "v", "n_iter", "n_solve", "alpha_index")
    for k in range(3):
        one = engine.run_sweep(prob, G[k:k + 1], alpha)
        sel = torch.as_tensor(np.nonzero(which == k)[0], device="cuda")
        for f in fields:
            got = getattr(res, f)[sel]
            assert torch.equal(got, getattr(one, f).expand_as(got)), (k, f)
    assert bool((res.status & 1).all())
    print("\nROW %s spectra/CTA=%.2f (B=%d, %d CTAs, %d SMs)" % (_name(c), B / grid, B, grid, sms))


@pytest.mark.gpu
@pytest.mark.parametrize("c", ONE_ALPHA, ids=_name)
def test_one_alpha(torch_cuda, c):
    """n_alpha = 1 against the oracle (same contract and checks as above), and the analyzers' results for one alpha:
    LineFit, Chi2Curvature and Entropy have no pick (-1, NaN rows; the reference raises on an all-NaN slice), Classic
    picks the only alpha (A_out bit for bit A[0]), Bryan averages one spectrum with weight 1."""
    res, o, wA, wc = _run_case(torch_cuda, c, "normal", 1, probability=True)
    idx = res.alpha_index[0].cpu().numpy()
    Aout, A = res.A_out[0].cpu().numpy(), res.A[0, 0].cpu().numpy()
    assert idx.tolist() == [-1, -1, -1, 0, 0], idx
    assert np.all(np.isnan(Aout[:3]))
    assert np.array_equal(Aout[3], A)
    np.testing.assert_allclose(Aout[4], A, rtol=1e-12, atol=0)
    p = res.logp[0].cpu().numpy()
    assert np.all(np.abs(p - o["probability"]) <= 1e-6 * np.abs(o["probability"])), (p, o["probability"])
    print("\nROW %s one-alpha dA/tol=%.3g dchi2/tol=%.3g" % (_name(c), wA, wc))
