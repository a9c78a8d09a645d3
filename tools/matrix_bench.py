"""Batched matrix continuation at the benchmark shape: B complex Hermitian 2x2 G(tau) (n_tau 2000, n_omega 1000,
60 alphas, cut 1e-11, sigma 1e-4; batched_matrix.synthetic_matrix_batch, fixed seed) through BatchedPoormanMaxEnt, next to
BatchedTauMaxEnt on the same number of scalar spectra at the same shape and the drop-in PoormanMaxEnt looped over a few
of the matrices.  Everything is timed in one process; the card's name and power limit are read in the same run.

    python tools/matrix_bench.py [--B 4096] [--loop 32] [--out profiles/r03_matrix_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--loop", type=int, default=32)
    ap.add_argument("--n_tau", type=int, default=2000)
    ap.add_argument("--n_omega", type=int, default=1000)
    ap.add_argument("--n_alpha", type=int, default=60)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join("profiles", "r03_matrix_bench.json"))
    a = ap.parse_args()
    import torch
    import maxent_b200 as mb
    from maxent_b200 import batched_matrix as bm
    if not torch.cuda.is_available():
        raise SystemExit("matrix_bench needs a CUDA device")
    tau, omega, G = bm.synthetic_matrix_batch(a.n_tau, a.n_omega, a.B, seed=7)
    alpha = mb.LogAlphaMesh(0.01, 2000.0, a.n_alpha)                 # the alpha mesh of bench.py
    cut, sigma = 1e-11, 1e-4

    job = mb.BatchedPoormanMaxEnt(use_hermiticity=True, use_complex=True, reduce_singular_space=cut)
    job.set_G_tau_data(tau, torch.from_numpy(G).cuda())
    job.omega, job.alpha_mesh = omega, alpha
    job.set_error(sigma)
    job.run_device()                                                # warm-up: problems, modules, workspaces
    torch.cuda.synchronize()
    n_elem = None
    runs = []
    for _ in range(a.reps):
        tl = []
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        plans, res, _, _ = job.run_device(timeline=tl)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        n_elem = int(len(plans[0]) + len(plans[1]))
        ms = lambda i, j: tl[i].elapsed_time(tl[j])
        # events: before pass 1, after pass 1, after the gather of the pass-2 rows, after the default models, after pass 2
        runs.append(dict(two_pass_s=ms(0, 4) / 1e3, pass1_s=ms(0, 1) / 1e3, default_models_step_s=ms(2, 3) / 1e3,
                         gap_between_passes_s=ms(1, 3) / 1e3, pass2_s=ms(3, 4) / 1e3, host_wall_s=wall))
    best = min(runs, key=lambda r: r["two_pass_s"])
    # the kernel alone: torch.ops.maxent_b200.poorman_models on pass 1's output of the last run, its arguments prepared
    # beforehand (CUDA events over repeated launches; each launch includes the 2 x 4 bytes per spectrum of index upload)
    from maxent_b200 import ops
    M = 2
    off = plans[1]
    A_out = res[0].A_out
    prob = job.maxent_offdiagonal.prepare()
    rows = torch.from_numpy(np.stack([off[:, 0] * M + off[:, 1], off[:, 0] * M + off[:, 2]], axis=1).astype(np.int32))
    P, ld = len(off), (prob.n_omega + 1) & ~1
    D = torch.empty((P, ld), dtype=torch.float64, device=A_out.device)
    v0 = torch.empty((P, prob.n_sv), dtype=torch.float64, device=A_out.device)
    ok = torch.empty((P,), dtype=torch.int32, device=A_out.device)
    Vp = prob.Vp[None].contiguous()

    def op():
        ops.poorman_models(A_out, 0, rows, prob.delta, 1e-6, None, Vp, None, D, v0, ok)
    op()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n_rep = 50
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n_rep):
        op()
    e1.record()
    e1.synchronize()
    op_alone = e0.elapsed_time(e1) / n_rep / 1e3

    # BatchedTauMaxEnt on the same number of scalar spectra at the same shape
    scal = mb.BatchedTauMaxEnt(reduce_singular_space=cut)
    Gs = mb.batched.synthetic_bootstrap_batch(a.n_tau, a.n_omega, n_elem, sigma=sigma).cuda()
    scal.set_G_tau_data(tau, Gs)
    scal.omega, scal.alpha_mesh = omega, alpha
    scal.set_error(sigma)
    scal.run_device(Gs, skip_small=True)
    scal_t = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        e0.record()
        scal.run_device(Gs, skip_small=True)
        e1.record()
        e1.synchronize()
        scal_t.append(e0.elapsed_time(e1) / 1e3)

    # the drop-in, one matrix at a time
    from maxent_b200.logtaker import VerbosityFlags

    def dropin(b):
        pm = mb.PoormanMaxEnt(use_hermiticity=True, use_complex=True, reduce_singular_space=cut)
        pm.set_verbosity(VerbosityFlags.Quiet)
        pm.set_G_tau_data(tau, G[b])
        pm.omega, pm.alpha_mesh = omega, alpha
        pm.set_error(sigma)
        return pm.run()
    dropin(0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b in range(a.loop):
        dropin(b)
    torch.cuda.synchronize()
    loop_s = (time.perf_counter() - t0) / a.loop

    out = dict(workload="BatchedPoormanMaxEnt, B=%d complex Hermitian 2x2, n_tau %d, n_omega %d, %d alphas, cut %g, "
                        "sigma %g, seed 7" % (a.B, a.n_tau, a.n_omega, a.n_alpha, cut, sigma),
               card=card(), element_spectra=n_elem, spectra_pass1=int(len(plans[0])), spectra_pass2=int(len(plans[1])),
               two_pass_device_s=best["two_pass_s"], element_spectra_per_s=n_elem / best["two_pass_s"],
               pass1_s=best["pass1_s"], pass2_s=best["pass2_s"], gap_between_passes_s=best["gap_between_passes_s"],
               default_models_step_in_job_s=best["default_models_step_s"], poorman_models_op_s=op_alone,
               notes="default_models_step_in_job_s: the whole default-model step between the passes (error plan, index "
                     "check on the host and upload, mx_poorman_models, masking of the skipped rows); poorman_models_op_s: "
                     "the operator alone; gap_between_passes_s: end of pass 1 to start of pass 2 (device events)",
               runs=runs,
               batched_tau_same_count_s=min(scal_t), batched_tau_spectra_per_s=n_elem / min(scal_t),
               dropin_poorman_per_matrix_s=loop_s, dropin_matrices_looped=a.loop,
               dropin_estimate_for_B_s=loop_s * a.B,
               n_sv=int(job.maxent_diagonal.prepare().n_sv))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
