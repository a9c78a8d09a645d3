#!/usr/bin/env python
"""Headline benchmark: spectra/sec for the full 60-alpha MaxEnt loop in FP64 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR]

A "step" is one pass of the hot path (data projection -> fused alpha sweep -> analyzers) over one
synthetic bootstrap batch: per GPU, `--spectra` (default 8192 = BASELINE config 5's per-GPU shard of the
65,536-spectrum batch) spectra with n_tau=2000, n_omega=1000, 60 alphas, reduce_singular_space=1e-11
(SURVEY.md 8(d) C5 recipe).  Weak scaling: every rank owns its own shard, no data-path collective.
The one collective of a multi-GPU job -- the NCCL gather of alpha_index / chi2 / A_out to rank 0 -- happens once per
job, after the last step: it is timed separately (`config.final_gather_ms_once_per_job`) and `e2e_job` reports the
throughput of a one-step job INCLUDING it.

One JSON line is printed by rank 0 (see the contract in the task statement).  `value` = device-resident
throughput, `e2e` = through the public batched API with pinned-host inputs/outputs, `roofline` = the
sweep kernel's achieved algorithmic FP64 FLOP/s against the FP64 peak MEASURED IN THIS RUN (mx_fp64_peak: DMMA and DFMA
saturating every SM, clocks sampled beside it), `cpu_baseline` = the oracle port of the reference timed on the host
cores in the same run (rank 0, N=1).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "spectra/sec (full 60-alpha MaxEnt loop, FP64)"
UNIT = "spectra/s"
# FP64 peak of this pool's B200 if the in-run measurement fails (tools/fp64_microbench.cu -> profiles/r01_fp64_microbench.json,
# DMMA m8n8k4 and DFMA both saturate at 37.0 TFLOP/s).  MEASURED_PEAKS.json holds no FP64 figure.
FP64_PEAK_FALLBACK_TFLOPS = 37.0
# DRAM traffic of the sweep kernel from the ncu capture under profiles/ (bytes read + written, per spectrum)
NCU_DRAM_BYTES_PER_SPECTRUM = int((6.98624e6 + 3.076533e9) / 296)   # profiles/r02c_sweep2_ncu_full_summary.json


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--spectra", type=int, default=8192, help="spectra per GPU and step")
    ap.add_argument("--n-tau", type=int, default=2000)
    ap.add_argument("--n-omega", type=int, default=1000)
    ap.add_argument("--n-alpha", type=int, default=60)
    ap.add_argument("--thr", type=float, default=1e-11, help="reduce_singular_space")
    ap.add_argument("--cost-function", default="normal", choices=["normal", "plusminus", "bryan"],
                    help="secondary measurements only: the headline metric is the default (normal) cost function")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-procs", type=int, default=0)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64, under 64 MB: "
                         "a fixed, seeded sample of the spectra)")
    return ap.parse_args()


def workload_name(a):
    return "bootstrap batch C5 shard: %d spectra/GPU, n_tau=%d, n_omega=%d, %d alphas, cut %g%s" % (
        a.spectra, a.n_tau, a.n_omega, a.n_alpha, a.thr,
        "" if a.cost_function == "normal" else ", cost function " + a.cost_function)


# --------------------------------------------------------------------------------------------------
# clocks
# --------------------------------------------------------------------------------------------------
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for n, v in zip(names, r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------------
# reference arm / CPU baseline
# --------------------------------------------------------------------------------------------------
def cpu_baseline(a, spectra=None, procs=None):
    procs = procs or a.cpu_procs or (os.cpu_count() or 1)
    spectra = spectra or procs
    cmd = [sys.executable, "-m", "oracle.cpu_baseline", "--n-tau", str(a.n_tau), "--n-omega", str(a.n_omega),
           "--n-alpha", str(a.n_alpha), "--spectra", str(spectra), "--procs", str(procs), "--thr", str(a.thr)]
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True)
    if out.returncode != 0:
        raise RuntimeError("cpu baseline failed: " + out.stderr[-2000:])
    return json.loads(out.stdout.strip().splitlines()[-1])


def cpu_baseline_block(r):
    return {"value": r["spectra_per_s"], "unit": UNIT, "cores": r["cores"], "kind": "port",
            "sample": "first %d spectra of the batch, full alpha loop, one process per spectrum x %d BLAS thread "
                      "(oracle/maxent_oracle.py = numpy port pinned bit-identically to TauMaxEnt.run; K^T W K setup "
                      "through BLAS); wall %.1f s; per-spectrum %.1f-%.1f s; LM iterations %d-%d; n_sv=%d"
                      % (r["spectra"], r["blas_threads"], r["wall_s"], min(r["per_spectrum_s"]),
                         max(r["per_spectrum_s"]), min(r["n_iter"]), max(r["n_iter"]), r["n_sv"])}


def run_reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    budget = float(os.environ.get("MAXENT_REF_BUDGET_S", "420"))
    t_begin = time.time()
    small = argparse.Namespace(**vars(a))
    small.n_tau, small.n_omega = 200, 100
    for _ in range(a.warmup):            # warm-up: process pool + BLAS on a small kernel (a full-size step is ~1 min)
        cpu_baseline(small)
    rows = []
    for k in range(a.steps):
        rows.append(cpu_baseline(a))
        if time.time() - t_begin > budget and k + 1 < a.steps:
            break
    n = sum(r["spectra"] for r in rows)
    wall = sum(r["wall_s"] for r in rows)
    val = n / wall
    merged = dict(rows[-1])
    merged.update(spectra_per_s=val)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus,
            "steps": len(rows), "steps_requested": a.steps, "warmup": a.warmup,
            "ms_per_step": 1000.0 * wall / len(rows), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a), "note": "CPU arm: each step = one bounded sample (cores spectra); "
                       "warm-up steps use a 200x100 kernel; stops early after MAXENT_REF_BUDGET_S=%g s" % budget},
            "cpu_baseline": cpu_baseline_block(merged),
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# native arm
# --------------------------------------------------------------------------------------------------
def algorithmic_flops(n_iter, n_q, n_s, n_alpha_total, n_omega, s, probability):
    """FP64 FLOPs of the singular-space algorithm the kernel implements (DESIGN.md, 'roofline'):
       per cost-function evaluation F_Q = 4 n_omega s + 8 n_omega   (x = V v, y = V^T H, pointwise exp/entropy)
       per LM iteration             F_H = n_omega s^2 + 2 s^3 + 4 s^2  (symmetric half of Z, J = Z Lambda Z + alpha Z, f = Z u)
       per solve                    F_S = s^3 / 3 + 2 s^2
    The survey's figure (section 8(d)) adds 2 n_tau s per evaluation for r = U Sigma y - G, which this
    formulation does not need (chi2 is diagonal in the rotated basis); it is reported as flops_survey."""
    FQ = 4.0 * n_omega * s + 8.0 * n_omega
    FH = n_omega * s * s + 2.0 * s ** 3 + 4.0 * s * s
    FS = s ** 3 / 3.0 + 2.0 * s * s
    F = n_iter * FH + n_q * FQ + n_s * FS
    if probability:
        F += n_alpha_total * (n_omega * s * s + s ** 3 / 3.0)
    return F


DUMP_BYTES = 60 * 10 ** 6          # data of --dump-outputs: under 64 MB with the .npy headers
DUMP_ANALYZERS = 3                 # LineFit, Chi2Curvature, Entropy: Classic and Bryan need the probability (not computed)


def dump_outputs(res, out_dir):
    """Write the result of one device-resident step (engine.SweepResult) to out_dir/<name>.npy in float64, so that two
    builds can be compared output for output: ``alpha`` and, for a fixed seeded sample of the batch (``spectrum_index``,
    as many spectra as fit in DUMP_BYTES), ``chi2``, ``S``, ``Q`` [n, n_alpha], ``alpha_index`` [n, 3], ``A_out``
    [n, 3, n_omega] and ``A`` [n, n_alpha, n_omega].  The solver's counters (n_iter, status, ...) describe how a result
    was reached rather than the result, and this path computes no probability (``logp``, Classic and Bryan analyzers):
    neither is written.  In a multi-GPU job rank 0 writes its own shard."""
    import numpy as np
    import torch
    B, n_alpha, n_omega = res.A.shape
    n_an = DUMP_ANALYZERS
    per_spectrum = 8 * (1 + 3 * n_alpha + n_an + n_an * n_omega + n_alpha * n_omega)
    n = min(B, (DUMP_BYTES - 8 * n_alpha) // per_spectrum)
    rows = np.sort(np.random.default_rng(0).choice(B, n, replace=False))
    idx = torch.as_tensor(rows, device=res.A.device)
    arrays = {"alpha": res.alpha, "spectrum_index": torch.as_tensor(rows), "alpha_index": res.alpha_index[idx, :n_an],
              "A_out": res.A_out[idx, :n_an]}
    for name in ("chi2", "S", "Q", "A"):
        arrays[name] = getattr(res, name)[idx]
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(np.float64))


def run_native(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from maxent_b200 import engine, batched

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # stdout carries the one JSON line: whatever the libraries print while the job runs (the NCCL version banner is
    # written straight to file descriptor 1) goes to stderr; the descriptor is restored just before the line is printed
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    # ---- the job: one BatchedTauMaxEnt per rank over its shard of the bootstrap batch ------------
    B = a.spectra
    job = batched.BatchedTauMaxEnt(cost_function=a.cost_function, reduce_singular_space=a.thr, device=dev)
    G_host = batched.synthetic_bootstrap_batch(a.n_tau, a.n_omega, B, first=rank * B, seed=5, pin=True)
    job.set_kernel_tau(np.linspace(0.0, 40.0, a.n_tau), batched.hyperbolic_omega(-10.0, 10.0, a.n_omega), beta=40.0)
    job.set_alpha_mesh_log(0.01, 2000.0, a.n_alpha)
    job.set_error(1.e-4)
    torch.zeros(1, device=dev)                      # CUDA context and library load are not kernel set-up
    torch.cuda.synchronize()
    t0 = time.time()
    job.prepare()                                   # kernel fill, truncated SVD, truncation, V' layout (once per kernel)
    torch.cuda.synchronize()
    setup_first_s = time.time() - t0                # includes the first-use costs of the library (module load, allocator)
    job.problem = None
    t0 = time.time()
    job.prepare()
    torch.cuda.synchronize()
    setup_s = time.time() - t0
    prob = job.problem

    G_dev = G_host.to(dev)
    torch.cuda.synchronize()
    import hashlib
    g_sha = hashlib.sha256(G_host[:min(B, 64)].numpy().tobytes()).hexdigest()[:16]

    # ---- FP64 peak of THIS device in THIS run (roofline denominator), clocks sampled while it runs --------------
    peak_meas = None
    try:
        from maxent_b200 import _lib
        lib = _lib.load()
        scratch = torch.empty((2 * 148 * 256 * 2,), dtype=torch.float64, device=dev)
        ps = ClockSampler(local)
        ps.start()
        t_dmma, t_dfma = ctypes.c_double(0.0), ctypes.c_double(0.0)
        t_pk = time.time()
        best = [0.0, 0.0]
        while True:                                 # ~1.5 s, so that the clock sampler sees the pipe under this load
            rc = lib.mx_fp64_peak(ctypes.byref(t_dmma), ctypes.byref(t_dfma), ctypes.c_void_p(scratch.data_ptr()),
                                  ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
            best = [max(best[0], t_dmma.value), max(best[1], t_dfma.value)]
            if rc != 0 or time.time() - t_pk > 1.5:
                break
        t_dmma.value, t_dfma.value = best
        pc = ps.stop()
        if rc == 0 and t_dmma.value > 1.0:
            peak_meas = {"dmma_tflops": t_dmma.value, "dfma_tflops": t_dfma.value, "sm_mhz": pc.get("sm_mhz"),
                         "reasons": pc.get("reasons")}
    except Exception as e:                      # keep the run alive, say so in the line
        peak_meas = {"error": str(e)}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident steps ---------------------------------------------------------------------
    for _ in range(a.warmup):
        res = job.run_device(G_dev)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(a.steps):
        res = job.run_device(G_dev)
    ev1.record()
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop()

    # ---- the dominant kernel alone (CUDA events around mx_alpha_sweep on the launching stream) ------
    k_ms = []
    for _ in range(max(1, min(a.steps, 3))):
        k_ms.append(job.time_sweep_kernel(G_dev))
    kernel_ms = sum(k_ms) / len(k_ms)
    n_iter = int(res.n_iter.sum()); n_q = int(res.n_qeval.sum()); n_s = int(res.n_solve.sum())
    n_trial = int(res.n_trial.sum()); n_batch = int(res.n_batch.sum())
    s = prob.n_sv
    flops = algorithmic_flops(n_iter, n_q, n_s, B * a.n_alpha, a.n_omega, s, False)
    flops_survey = flops + n_q * 2.0 * a.n_tau * s
    peak = FP64_PEAK_FALLBACK_TFLOPS
    peak_src = "fallback: FP64 DMMA/DFMA peak of this pool's B200 measured in round 1, profiles/r01_fp64_microbench.json"
    if peak_meas and "dmma_tflops" in peak_meas:
        peak = max(peak_meas["dmma_tflops"], peak_meas["dfma_tflops"])
        peak_src = ("measured in this run on this device (mx_fp64_peak: every SM saturated with DMMA m8n8k4 / DFMA chains; "
                    "MEASURED_PEAKS.json has no FP64 entry)")
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        for key in ("fp64_tflops", "dmma_tflops"):
            if key in mp:
                peak, peak_src = float(mp[key]), "MEASURED_PEAKS.json:" + key
    except Exception:
        pass
    achieved = flops / (kernel_ms * 1e-3) / 1e12

    # ---- end to end through the public API: pinned host G in, pinned host results out ---------------
    for _ in range(max(1, min(a.warmup, 2))):
        out = job.run(G_host)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        out = job.run(G_host)
    e1.record()
    barrier()
    e2e_ms = e0.elapsed_time(e1)
    h2d, d2h = out.h2d_bytes, out.d2h_bytes

    # ---- what the OPTIONAL copy of every A_alpha(omega) to the host would cost (the reference keeps them all in
    #      memory; the batched API leaves them on the device: BatchedMaxEntResult.A(b)) -- measured once on a slice ----
    nb_a = min(B, 1024)
    a_pin = torch.empty((nb_a,) + tuple(out.device.A.shape[1:]), dtype=torch.float64, pin_memory=True)
    torch.cuda.synchronize()
    ea0, ea1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ea0.record()
    a_pin.copy_(out.device.A[:nb_a], non_blocking=True)
    ea1.record()
    torch.cuda.synchronize()
    full_A_ms = ea0.elapsed_time(ea1) * (B / nb_a)
    full_A_bytes = B * out.device.A.shape[1] * out.device.A.shape[2] * 8
    del a_pin

    # ---- max over ranks -------------------------------------------------------------------------------
    gather_ms = 0.0
    if world > 1:
        # the one collective of the job: gather the analyzer outputs on rank 0 (NCCL over NVLink), once per job
        batched.gather_results(out, dst=0)              # first call sets up the NCCL connections
        barrier()
        t_g = time.time()
        gathered = batched.gather_results(out, dst=0)
        barrier()
        gather_ms = (time.time() - t_g) * 1e3
        if rank == 0:
            assert gathered["alpha_index"].shape[0] == world * B
    t = torch.tensor([dev_ms, e2e_ms, kernel_ms, gather_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    # the roofline block pairs rank 0's own kernel time with rank 0's own FLOP counters; the job times are the maxima
    dev_ms, e2e_ms, _, gather_ms = [float(x) for x in t.tolist()]

    if rank == 0:
        total = world * B * a.steps
        value = total / (dev_ms * 1e-3)
        e2e = total / (e2e_ms * 1e-3)
        idx = res.alpha_index.cpu().numpy()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": dev_ms / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(a), "n_sv": s, "parallelism": "spectra sharded x%d, no data-path collective" % world,
                       "l2": "inputs/outputs larger than L2 (G %.0f MB, A(alpha) %.1f GB per step); V' (%.0f KB) is L2-resident by design"
                             % (B * a.n_tau * 8 / 1e6, B * a.n_alpha * a.n_omega * 8 / 1e9, prob.Vt.numel() * 8 / 1e3),
                       "final_gather_ms_once_per_job": round(gather_ms, 3), "G_sha256_first_64_rows": g_sha,
                       "optional_full_A_alpha_d2h": {"bytes_per_step": full_A_bytes, "ms_per_step_extrapolated": round(full_A_ms, 1),
                                                     "note": "not part of e2e: A_alpha stays on the device, e2e returns A_out of the five analyzers"},
                       "setup_s_once_per_kernel": round(setup_s, 3), "setup_s_first_call": round(setup_first_s, 3),
                       "svd": getattr(prob, "svd_sweeps", None),
                       "spectra_per_cta": prob.config["spectra_per_cta"], "smem_bytes": prob.config["smem_bytes"],
                       "lm_iterations_per_spectrum": n_iter / B, "q_evals_per_spectrum": n_q / B, "solves_per_spectrum": n_s / B,
                       "device_trials_per_lm_iteration": n_trial / max(n_iter, 1),
                       "device_batches_per_lm_iteration": n_batch / max(n_iter, 1),
                       "converged_frac": float((res.status & 1).double().mean()),
                       "linefit_idx_hist": {int(k): int(v) for k, v in zip(*np.unique(idx[:, 0], return_counts=True))},
                       "chi2curv_idx_hist": {int(k): int(v) for k, v in zip(*np.unique(idx[:, 1], return_counts=True))}},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms / a.steps},
            "e2e_job": {"value": world * B / ((e2e_ms / a.steps + gather_ms) * 1e-3), "unit": UNIT,
                        "what": "one end-to-end step followed by the final gather of alpha_index / chi2 / A_out to rank 0 "
                                "(a complete %d-spectrum job)" % (world * B)},
            "gpu_launches": a.steps * job.launches_per_step,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                         "traffic": NCU_DRAM_BYTES_PER_SPECTRUM * B, "traffic_unit": "bytes per launch",
                         "traffic_source": "ncu --set full dram__bytes_read.sum + dram__bytes_write.sum of one 296-spectrum "
                                           "launch (profiles/r02c_*), scaled to this launch's spectra; algorithmic bytes per spectrum = "
                                           "G in + A(alpha) out = %d" % (a.n_tau * 8 + a.n_alpha * a.n_omega * 8),
                         "traffic_note": "accepted: %.0fx the algorithmic bytes = ~23 GB/s, 0.3 %% of the HBM bandwidth (the kernel is "
                                         "FP64-pipe bound).  It is write-back of L2 lines, not re-reads: the solver's register spills "
                                         "(128-register cap for two CTAs per SM; 58 GB of local-memory stores per 296-spectrum wave "
                                         "into L2) and the per-CTA scratch rows of w = dH/dx share the L2 with the streamed A(alpha) "
                                         "output, and ~5 %% of those lines are evicted dirty"
                                         % (NCU_DRAM_BYTES_PER_SPECTRUM / (a.n_tau * 8 + a.n_alpha * a.n_omega * 8)),
                         "peak_measured_in_run": peak_meas,
                         "kernel": "mx2::sweep2_kernel", "kernel_ms": kernel_ms,
                         "kernel_share_of_step": kernel_ms / (dev_ms / a.steps),
                         "flops_per_launch": flops, "flops_per_spectrum": flops / B,
                         "flops_survey_formula_per_spectrum": flops_survey / B,
                         "frac_with_survey_formula": flops_survey / (kernel_ms * 1e-3) / 1e12 / peak,
                         "pipe": "FP64 (DMMA m8n8k4 + DFMA share one pipe on B200)", "peak_source": peak_src},
        }
        if a.dump_outputs:
            dump_outputs(res, a.dump_outputs)
        if world == 1 and not a.no_cpu_baseline and a.cost_function == "normal":
            try:
                line["cpu_baseline"] = cpu_baseline_block(cpu_baseline(a))
            except Exception as e:        # the GPU numbers stay valid; say why the CPU leg is missing
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %s" % e}
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line))
        sys.stdout.flush()
    if world > 1:
        dist.destroy_process_group()


def main():
    a = parse_args()
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_native(a)


if __name__ == "__main__":
    main()
