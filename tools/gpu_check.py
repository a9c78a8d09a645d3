"""GPU diagnostic: run the fused sweep on the golden fixtures and print parity metrics vs the reference outputs."""
import os, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from maxent_b200 import engine
from oracle import maxent_oracle as mo

np.set_printoptions(linewidth=220, precision=2)
names = sys.argv[1:] or ["g2_synth_200x100.npz", "g3_plusminus_offdiag.npz", "g4_bryan_200x100.npz",
                         "g1_semicircular_prob.npz", "g5_config1_cut1e-11.npz"]
svd = os.environ.get("MX_SVD", "jacobi")
for name in names:
    g = dict(np.load(os.path.join("tests/golden", name)))
    K = mo.tau_kernel(g["tau"], g["omega"], None)
    delta = mo.omega_delta(g["omega"]); D = mo.flat_default_model(g["omega"])
    t0 = time.time()
    prob = engine.SharedProblem(K, g["err"], D, delta, variant=str(g["variant"]),
                                reduce_singular_space=float(g["reduce_singular_space"]), svd=svd)
    torch.cuda.synchronize(); t1 = time.time()
    res = engine.run_sweep(prob, g["G"], g["ref_alpha"], probability=bool(g["use_probability"]))
    torch.cuda.synchronize(); t2 = time.time()
    chi2 = res.chi2[0].cpu().numpy(); A = res.A[0].cpu().numpy(); S = res.S[0].cpu().numpy()
    print("==", name, "n_sv", prob.n_sv, "ref", int(g["ref_n_sv"]), "cfg", prob.config, "prep %.3fs sweep %.3fs" % (t1 - t0, t2 - t1),
          "svd_sweeps", getattr(prob, "svd_sweeps", None))
    Sref = g["ref_K_S"]; Sg = prob.S.cpu().numpy()
    n = min(len(Sref), len(Sg))
    print("  max rel diff singular values:", np.max(np.abs(Sg[:n] / Sref[:n] - 1)))
    print("  rel chi2", np.abs(chi2 / g["ref_chi2"] - 1))
    print("  rel A   ", np.max(np.abs(A - g["ref_A"]), axis=1) / np.max(np.abs(g["ref_A"]), axis=1))
    print("  rel S   ", np.abs(S / g["ref_S"] - 1))
    print("  n_iter", res.n_iter[0].cpu().numpy(), "sum", int(res.n_iter.sum()), "nq", int(res.n_qeval.sum()), "ns", int(res.n_solve.sum()))
    print("  conv", res.status[0].cpu().numpy())
    if bool(g["use_probability"]):
        print("  logp", res.logp[0].cpu().numpy(), "ref", g["ref_probability"])
    idx = res.alpha_index[0].cpu().numpy()
    print("  analyzers idx", idx, "ref", [int(g.get("ref_idx_" + k, -1)) for k in
          ("LineFitAnalyzer", "Chi2CurvatureAnalyzer", "EntropyAnalyzer", "ClassicAnalyzer")])
