import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["MAXENT_B200_LIB"] = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "maxent_b200/libmaxent_b200_tprof.so")
import numpy as np, torch
from maxent_b200 import batched, engine
job = batched.BatchedTauMaxEnt(reduce_singular_space=1e-11)
G = batched.synthetic_bootstrap_batch(2000, 1000, 592, seed=5)
job.set_kernel_tau(np.linspace(0.0, 40.0, 2000), batched.hyperbolic_omega(-10.0, 10.0, 1000), beta=40.0)
job.set_alpha_mesh_log(0.01, 2000.0, 60); job.set_error(1.e-4)
prob = job.prepare(); Gd = G.cuda()
for cap, n in (("99", 592), ("1", 148)):
    os.environ["MX_MAX_CTAS_PER_SM"] = cap
    r = engine.run_sweep(prob, Gd[:n], job.alpha_effective(), want_v=False, analyze_results=False, phase_timers=True)
    torch.cuda.synchronize()
    pf = r.phase_cycles.double().cpu().numpy().sum(0)
    print(json.dumps(dict(cap=cap, steps=pf[2], empty_wait_clk_per_step=pf[0]/pf[2], full_wait_clk_per_step=pf[1]/pf[2],
          waited_frac=pf[5]/pf[2], latency_when_waited_clk=pf[4]/max(pf[5],1))))
