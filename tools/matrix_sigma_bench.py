"""Batched matrix-valued self-energy continuation at the benchmark shape: B = 4096 complex Hermitian 2x2 self-energies
Sigma_b(i omega_n) (beta 40, n_iw 1000), n_omega 1000 hyperbolic on [-10, 10], 60 alphas from 0.01 to 2000, cut 1e-11,
sigma 1e-4, back to n_w = 2000 real frequencies on [-10, 10] at eta = 0.01 through BatchedSigmaContinuator with
maxent=BatchedPoormanMaxEnt(use_complex=True) (inversion).  Sigma_b = U_b diag(t_bm^2 g_sc(i omega_n; t_bm)) U_b^dagger
(matrix Bethe lattice, t in [0.8, 1.2], random unitary U_b) plus complex noise of size sigma on every element, fixed seed.

Times, all from CUDA events in one process:
* the forward resolvent G_aux = ((i nu + C) 1 - Sigma)^-1 (mx_matrix_resolvent mode 0) and the backward resolvent
  Sigma = (z + C) 1 - G_aux(z)^-1 (mode 1), each the mean over >= 20 launches after warm-up, out of place, with the bytes
  they must move (16 M^2 bytes read and written per (b, k)) over the time: achieved DRAM bytes/s.  Their working sets
  (2 x 262 MB and 2 x 524 MB) are larger than the 126 MB L2, so they stream from DRAM;
* pass 1, the Poorman default models and pass 2 of the continuation (BatchedElementwiseMaxEnt.run_device timeline);
* the device assembly of A_aux from the two passes and the Hilbert apply of every part, and the whole sigma_w call.
The card's name and power limit are read in the same run.

    python tools/matrix_sigma_bench.py [--B 4096] [--out profiles/r05_matrix_sigma_bench.json]
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


def events_ms(torch, fn, n):
    """Mean milliseconds of fn() over n launches, CUDA events on the current stream."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=4096)
    ap.add_argument("--M", type=int, default=2)
    ap.add_argument("--n_iw", type=int, default=1000)
    ap.add_argument("--n_omega", type=int, default=1000)
    ap.add_argument("--n_alpha", type=int, default=60)
    ap.add_argument("--n_w", type=int, default=2000)
    ap.add_argument("--eta", type=float, default=0.01)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--launches", type=int, default=20)
    ap.add_argument("--out", default=os.path.join("profiles", "r05_matrix_sigma_bench.json"))
    a = ap.parse_args()
    import torch
    import maxent_b200 as mb
    from maxent_b200 import ops, real_frequency
    from oracle import matrix_sigma as ms
    if not torch.cuda.is_available():
        raise SystemExit("matrix_sigma_bench needs a CUDA device")
    beta, sigma, cut, seed = 40.0, 1e-4, 1e-11, 23
    B, M = a.B, a.M
    nu = np.pi / beta * (2 * np.arange(a.n_iw) + 1)
    rng = np.random.default_rng(seed)
    t = 0.8 + 0.4 * rng.random((B, M))
    U = ms.random_unitary(B, M, seed + 1)
    S = ms.bethe_matrix_sigma(1j * nu, t, U)
    S = S + sigma * (rng.standard_normal(S.shape) + 1j * rng.standard_normal(S.shape))
    omega = mb.HyperbolicOmegaMesh(-10, 10, a.n_omega)
    w = np.linspace(-10, 10, a.n_w)

    sc = mb.BatchedSigmaContinuator(maxent=mb.BatchedPoormanMaxEnt(use_complex=True))
    sc.set_S_iw_data(nu, S)
    job = sc.maxent
    job.omega = omega
    job.alpha_mesh = mb.LogAlphaMesh(0.01, 2000.0, a.n_alpha)
    for wk in job._workers():
        wk.reduce_singular_space = cut
    job.set_error(sigma)

    # forward resolvent, out of place on the device-resident Sigma
    X = torch.as_tensor(S, device="cuda")
    z_iw = torch.complex(torch.zeros(a.n_iw, dtype=torch.float64), torch.as_tensor(nu)).cuda()
    C = torch.zeros(B, dtype=torch.float64, device="cuda")
    Y = torch.empty_like(X)
    fwd = lambda: ops.matrix_resolvent(X, z_iw, C, 0, Y)
    for _ in range(3):
        fwd()
    fwd_ms = events_ms(torch, fwd, a.launches)
    fwd_bytes = 2 * 16 * M * M * B * a.n_iw

    t0 = time.perf_counter()
    res = sc.run()                                                   # warm-up: kernel fill, SVD, modules, workspaces
    torch.cuda.synchronize()
    first_run_s = time.perf_counter() - t0
    phases = []
    for _ in range(a.reps):
        tl = []
        torch.cuda.synchronize()
        job.run_device(timeline=tl)
        tl[-1].synchronize()
        phases.append([tl[i].elapsed_time(tl[i + 1]) / 1e3 for i in range(len(tl) - 1)])
    best = min(phases, key=sum)

    # sigma_w and its parts: assembly, Hilbert apply of every part, backward resolvent
    sc.sigma_w(w, a.eta)                                            # builds and caches the table
    torch.cuda.synchronize()
    asm_ms = events_ms(torch, lambda: res.A_out_device(0), a.launches)
    A = res.A_out_device(0)
    n_rows = int(A.numel() // a.n_omega)
    Mt, w_d = real_frequency.hilbert_table(np.asarray(omega), w, a.eta)
    A2 = A.reshape(n_rows, a.n_omega)
    apply_ms = events_ms(torch, lambda: real_frequency._apply(A2, Mt, w_d, a.eta, 0), a.launches)
    Xw = sc.sigma_w(w, a.eta).clone()                               # the resolvent's cost does not depend on the values
    z_w = torch.complex(w_d, torch.full_like(w_d, a.eta))
    Yw = torch.empty_like(Xw)
    bwd = lambda: ops.matrix_resolvent(Xw, z_w, C, 1, Yw)
    for _ in range(3):
        bwd()
    bwd_ms = events_ms(torch, bwd, a.launches)
    bwd_bytes = 2 * 16 * M * M * B * a.n_w
    sw_ms = events_ms(torch, lambda: sc.sigma_w(w, a.eta), 5)
    sw = sc.sigma_w(w, a.eta)
    finite = int(torch.isfinite(torch.view_as_real(sw)).reshape(B, -1).all(dim=1).sum())

    out = dict(
        workload="BatchedSigmaContinuator (inversion) with BatchedPoormanMaxEnt(use_complex=True): B=%d complex "
                 "Hermitian %dx%d Sigma, beta %g, n_iw %d, n_omega %d hyperbolic [-10, 10], %d alphas 0.01..2000, cut %g, "
                 "sigma %g; n_w %d linear [-10, 10], eta %g; seed %d"
                 % (B, M, M, beta, a.n_iw, a.n_omega, a.n_alpha, cut, sigma, a.n_w, a.eta, seed),
        card=card(),
        forward_resolvent_ms=fwd_ms, forward_resolvent_bytes=fwd_bytes,
        forward_resolvent_GB_per_s=fwd_bytes / fwd_ms / 1e6,
        pass1_ms=best[0] * 1e3, gather_pass2_rows_ms=best[1] * 1e3, default_models_ms=best[2] * 1e3,
        pass2_ms=best[3] * 1e3, continuation_ms=sum(best) * 1e3, continuation_runs_s=[sum(p) for p in phases],
        first_run_host_s=first_run_s,
        assembly_ms=asm_ms, hilbert_apply_ms=apply_ms, hilbert_apply_rows=n_rows,
        backward_resolvent_ms=bwd_ms, backward_resolvent_bytes=bwd_bytes,
        backward_resolvent_GB_per_s=bwd_bytes / bwd_ms / 1e6,
        sigma_w_call_ms=sw_ms, sigma_w_finite_matrices=finite,
        notes="CUDA events in one process.  Resolvent times: mean over %d out-of-place launches after 3 warm-up launches; "
              "bytes = 16 M^2 read + 16 M^2 written per (b, k); working sets larger than L2.  Continuation: "
              "run_device timeline (pass 1, gather of the pass-2 rows, Poorman default models, pass 2), best of %d.  "
              "assembly (A_out_device) and hilbert_apply (mode 0, every part of every element): mean over %d launches; "
              "sigma_w_call_ms: mean over 5 calls with the table cached." % (a.launches, a.reps, a.launches))
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
