#!/usr/bin/env python
"""Laplace vs Gaussian MMD kernel on one configs[1] sweep point (200 static episodes, beta noise 0.3, O = 4, np = 50, nr = 5), in one process:
the mmd_opt 200-episode solve with the two kernels alternating (CUDA events around each solve, 3 runs each after a warm-up), the device time
per kernel class of one staged solve (mpcmmd_profile_solve; the inner CEM is part of the risk class) and the inner-CEM kernels' time per
launch (torch.profiler), the batch-1 p50 latency, one nr = 10 and one nr = 20 point at a reduced episode count, the accepted-episode count
of each kernel and the collision / lane fractions of both kernels' plans under counter-based noise at 10^4 rollouts
(`validation.threefry_stats_batch`).  The GPU name and power limit are read in the same run.
usage: mmd_kernel_probe.py [OUT.json]   (prints the record; also writes it to OUT.json if given)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mpc-mmd_b200")):
    sys.path.insert(1, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402
import __graft_entry__ as G  # noqa: E402

G.build()
from mpcmmd_b200 import CEM, driver, scenes, validation as V  # noqa: E402

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
KEYS = ("idx_mpc", "init_state", "mean_param", "cov_param", "x_obs_traj", "y_obs_traj", "v_des")
KERNELS = ("laplace", "gaussian")
out = dict(gpu=gpu, workload="configs[1] sweep point: 200 static episodes, mmd_opt, beta noise 0.3, O = 4, np = 50, nr = 5")


def timed(prob, E, runs):
    host = scenes.static_batch(prob, list(range(E)), "static")
    dev = {k: torch.as_tensor(host[k], device="cuda:0") for k in KEYS}
    run = lambda: prob.solve_batch_device("mmd_opt", *[dev[k] for k in KEYS])
    ts = []
    for _ in range(runs):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); run(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
    return ts, run


def make(nr, E, kernel, **kw):
    return CEM(nr, 4, 0.3, 50, "beta", 0.0, 0.0, variant="static", max_episodes=E, kernel=kernel, **kw)


# 200-episode solve, kernels alternating
probs = {k: make(5, 200, k) for k in KERNELS}
runs = {k: timed(probs[k], 200, 1)[1] for k in KERNELS}          # warm-up (graph capture) of both
solve = {k: [] for k in KERNELS}
for _ in range(3):
    for k in KERNELS:
        solve[k] += timed(probs[k], 200, 1)[0]
out["solve_200_ms"] = solve
out["solve_200_ms_median"] = {k: float(np.median(v)) for k, v in solve.items()}
out["profile_solve"], out["inner_kernel_us_per_launch"] = {}, {}
for k in KERNELS:
    runs[k](); torch.cuda.synchronize()
    out["profile_solve"][k] = probs[k].profile_solve("mmd_opt", 200)
    with profile(activities=[ProfilerActivity.CUDA]) as pr:
        runs[k](); torch.cuda.synchronize()
    out["inner_kernel_us_per_launch"][k] = {e.key: round(e.device_time_total / max(e.count, 1), 1) for e in pr.key_averages()
                                             if "k_inner_cem" in e.key or "k_opt_risk" in e.key}
del probs, runs

# batch-1 latency
lat = {}
for k in KERNELS:
    p = make(5, 1, k)
    ts, _ = timed(p, 1, 23)
    lat[k] = float(np.percentile(ts[3:], 50))
out["batch1_p50_ms"] = lat

# other reduced-set sizes at a reduced episode count
out["other_nr"] = {}
for nr, E in ((10, 20), (20, 4)):
    rec = {}
    for k in KERNELS:
        p = make(nr, E, k)
        timed(p, E, 1)
        rec[k] = float(np.median(timed(p, E, 3)[0]))
    out["other_nr"]["nr%d_%dep_ms" % (nr, E)] = rec

# acceptance and Monte-Carlo collision / lane fractions of the plans (10^4 counter-based rollouts per trajectory)
import tempfile  # noqa: E402
tmp = tempfile.mkdtemp(prefix="mmd_kernel_probe_")
common = ["--noises", "beta", "--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "4", "--num_prime", "50",
          "--acc_const_noise", "0.0", "--steer_const_noise", "0.0", "--costs", "mmd_opt", "--num_configs", "200"]
out["plans"] = {}
for k in KERNELS:
    root = os.path.join(tmp, k)
    driver.run_sweep(driver.build_parser().parse_args(common + ["--root", root, "--kernel", k]), log=lambda *a: None)
    d = V._load(root, "beta", 0.3, 50, "mmd_opt", 5, 4)
    items = [V._item(d, i, i, False) for i in range(d["cx"].shape[0])]
    prob = make(5, 1, k)
    count, lane = V.threefry_stats_batch(prob, items, 50, 0.3, "beta", 4, n_roll=10000)
    out["plans"][k] = dict(accepted=int(d["cx"].shape[0]), mean_collision_fraction=float(np.mean(count) / 10000),
                           mean_lane_fraction=float(np.mean(lane) / 10000))

print(json.dumps(out, indent=1))
if len(sys.argv) > 1:
    json.dump(out, open(sys.argv[1], "w"), indent=1)
