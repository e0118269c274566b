#!/usr/bin/env python
"""Device time of one 200-episode configs[1] mmd_opt solve: 10 solves timed with CUDA events after 3 warm-up solves, then one solve under
torch.profiler (CUDA activities) for the time per kernel.  usage: solve_kernel_times.py [OUT.json]"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mpc-mmd_b200")):
    sys.path.insert(1, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402
import __graft_entry__ as G  # noqa: E402

G.build()
from mpcmmd_b200 import CEM, scenes  # noqa: E402

keys = ("idx_mpc", "init_state", "mean_param", "cov_param", "x_obs_traj", "y_obs_traj", "v_des")
E = 200
prob = CEM(5, 4, 0.3, 50, "beta", 0.0, 0.0, variant="static", max_episodes=E, device=0)
host = scenes.static_batch(prob, list(range(E)), "static")
dev_in = {k: torch.as_tensor(host[k], device="cuda:0") for k in keys}
run = lambda: prob.solve_batch_device("mmd_opt", *[dev_in[k] for k in keys])
for _ in range(3):
    run()
torch.cuda.synchronize()
ts = []
for _ in range(10):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); run(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
with profile(activities=[ProfilerActivity.CUDA]) as pr:
    run(); torch.cuda.synchronize()
kern = {}
for e in pr.key_averages():
    t = getattr(e, "device_time_total", 0)
    if t > 0:
        kern[e.key] = {"count": e.count, "avg_us": t / max(e.count, 1), "total_us": t}
out = {"gpu": torch.cuda.get_device_name(0), "solve_ms": ts, "solve_ms_median": float(np.median(ts)), "kernels_us": kern}
print(json.dumps({"solve_ms_median": out["solve_ms_median"], "k_inner_cem_fast_us": {k: round(v["avg_us"], 1) for k, v in kern.items() if "k_inner_cem" in k}}))
if len(sys.argv) > 1:
    json.dump(out, open(sys.argv[1], "w"), indent=1)
