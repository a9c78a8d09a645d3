"""Batched self-energy continuation at the benchmark shape: B = 8192 scalar self-energies Sigma_b(i omega_n)
(beta 40, n_iw 1000 = 2000 stacked rows, the n_tau of bench.py), n_omega 1000 hyperbolic on [-10, 10], 60 alphas from
0.01 to 2000, cut 1e-11, sigma 1e-4, back to n_w = 2000 real frequencies on [-10, 10] at eta = 0.01 through
BatchedSigmaContinuator (inversion).  Sigma_b = t_b^2 g_sc(i omega_n) (Bethe lattice, t_b in [0.8, 1.2]) plus noise,
fixed seed.

Times, all from CUDA events in one process: the device-resident auxiliary continuation, mx_hilbert_table, and
mx_hilbert_apply alone (>= 20 launches after warm-up, on the analyzer slot of A_out read in place) with its FLOP
(4 R n_omega n_w) over the DMMA peak that mx_fp64_peak measures in the same run.  A (65 MB) and the table (32 MB) fit the
L2 cache: the apply time is that of a warm L2, which is how the continuator calls it (right after the continuation).
The card's name and power limit are read in the same run.

    python tools/sigma_bench.py [--B 8192] [--out profiles/r04_sigma_bench.json]
"""
import argparse
import ctypes
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
    ap.add_argument("--B", type=int, default=8192)
    ap.add_argument("--n_iw", type=int, default=1000)
    ap.add_argument("--n_omega", type=int, default=1000)
    ap.add_argument("--n_alpha", type=int, default=60)
    ap.add_argument("--n_w", type=int, default=2000)
    ap.add_argument("--eta", type=float, default=0.01)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--apply_launches", type=int, default=50)
    ap.add_argument("--out", default=os.path.join("profiles", "r04_sigma_bench.json"))
    a = ap.parse_args()
    import torch
    import maxent_b200 as mb
    from maxent_b200 import _lib, ops, real_frequency
    if not torch.cuda.is_available():
        raise SystemExit("sigma_bench needs a CUDA device")
    beta, sigma, cut = 40.0, 1e-4, 1e-11
    nu = np.pi / beta * (2 * np.arange(a.n_iw) + 1)
    rng = np.random.default_rng(17)
    t = 0.8 + 0.4 * rng.random(a.B)
    z = 1j * nu
    g_sc = lambda tt: (z[None, :] - np.sqrt(z[None, :] - 2 * tt[:, None]) * np.sqrt(z[None, :] + 2 * tt[:, None])) / (
        2 * tt[:, None] ** 2)
    S = t[:, None] ** 2 * g_sc(t) + sigma * (rng.standard_normal((a.B, a.n_iw)) + 1j * rng.standard_normal((a.B, a.n_iw)))
    omega = mb.HyperbolicOmegaMesh(-10, 10, a.n_omega)
    w = np.linspace(-10, 10, a.n_w)

    sc = mb.BatchedSigmaContinuator(method="inversion")
    sc.maxent.reduce_singular_space = cut
    sc.set_S_iw_data(nu, S)
    sc.maxent.omega = omega
    sc.maxent.alpha_mesh = mb.LogAlphaMesh(0.01, 2000.0, a.n_alpha)
    sc.maxent.set_error(sigma)
    job = sc.maxent
    G_dev = torch.as_tensor(job.G, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    t0 = time.perf_counter()
    sc.run()                                                          # warm-up: kernel fill, SVD, modules, workspaces
    torch.cuda.synchronize()
    first_run_s = time.perf_counter() - t0
    cont = []
    for _ in range(a.reps):
        torch.cuda.synchronize()
        e0.record()
        res = job.run_device(G_dev, skip_small=True)
        e1.record()
        e1.synchronize()
        cont.append(e0.elapsed_time(e1) / 1e3)

    # mx_hilbert_table: once per (mesh, w, eta); timed on fresh buffers after one warm-up launch
    om_d = torch.as_tensor(np.asarray(omega), device="cuda")
    w_d = torch.as_tensor(w, device="cuda")
    M = torch.empty((a.n_w, a.n_omega), dtype=torch.complex128, device="cuda")
    ops.hilbert_table(om_d, w_d, a.eta, M)
    tab = []
    for _ in range(5):
        torch.cuda.synchronize()
        e0.record()
        ops.hilbert_table(om_d, w_d, a.eta, M)
        e1.record()
        e1.synchronize()
        tab.append(e0.elapsed_time(e1) / 1e3)

    # mx_hilbert_apply alone, mode 2 (inversion), on the LineFit slot of A_out in place
    A = res.A_out[:, 0, :]
    R = int(A.shape[0])
    shift = torch.zeros(R, dtype=torch.float64, device="cuda")
    out = torch.empty((R, a.n_w), dtype=torch.complex128, device="cuda")
    for _ in range(3):
        ops.hilbert_apply(A, M, w_d, a.eta, 2, None, shift, out)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(a.apply_launches):
        ops.hilbert_apply(A, M, w_d, a.eta, 2, None, shift, out)
    e1.record()
    e1.synchronize()
    apply_s = e0.elapsed_time(e1) / 1e3 / a.apply_launches
    flop = 4.0 * R * a.n_omega * a.n_w

    # the whole sigma_w call (table cached after the first call, NaN masking included)
    sc.sigma_w(w, a.eta)
    torch.cuda.synchronize()
    e0.record()
    sw = sc.sigma_w(w, a.eta)
    e1.record()
    e1.synchronize()
    sigma_w_s = e0.elapsed_time(e1) / 1e3
    ok_rows = int(torch.isfinite(sw.real).all(dim=1).sum())

    lib = _lib.load()
    dm, df = ctypes.c_double(), ctypes.c_double()
    scratch = torch.empty(2 * lib.mx_device_sm_count() * 256, dtype=torch.float64, device="cuda")
    _lib.check(lib.mx_fp64_peak(ctypes.byref(dm), ctypes.byref(df), ctypes.c_void_p(scratch.data_ptr()),
                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)), "mx_fp64_peak")
    apply_tflops = flop / apply_s / 1e12
    best = min(cont)
    out_json = dict(
        workload="BatchedSigmaContinuator (inversion), B=%d, beta %g, n_iw %d (%d stacked rows), n_omega %d hyperbolic "
                 "[-10, 10], %d alphas 0.01..2000, cut %g, sigma %g; n_w %d linear [-10, 10], eta %g; seed 17"
                 % (a.B, beta, a.n_iw, 2 * a.n_iw, a.n_omega, a.n_alpha, cut, sigma, a.n_w, a.eta),
        card=card(), n_sv=int(job.prepare().n_sv),
        continuation_device_s=best, continuation_runs_s=cont, continuation_spectra_per_s=a.B / best,
        first_run_host_s=first_run_s,
        hilbert_table_s=min(tab), hilbert_apply_s=apply_s, hilbert_apply_launches_timed=a.apply_launches,
        hilbert_apply_flop=flop, hilbert_apply_tflops=apply_tflops,
        fp64_peak_dmma_tflops=dm.value, fp64_peak_dfma_tflops=df.value,
        hilbert_apply_share_of_dmma_peak=apply_tflops / dm.value,
        hilbert_apply_share_of_continuation=apply_s / best,
        sigma_w_call_s=sigma_w_s, sigma_w_finite_rows=ok_rows,
        notes="continuation_device_s: BatchedTauMaxEnt.run_device on the device-resident stacked G_aux (project, sweep, "
              "analyze), CUDA events, best of the runs; hilbert_apply_s: mean over the timed launches after 3 warm-up "
              "launches, A and M resident in L2; share of peak = achieved FLOP/s over the DMMA rate mx_fp64_peak "
              "measured in this run")
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(out_json, f, indent=1)
    print(json.dumps(out_json))


if __name__ == "__main__":
    main()
