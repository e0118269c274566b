#!/usr/bin/env python
"""Monte-Carlo risk of solver plans against the solver's own few-sample estimates, on one configs[1] sweep point: 200 static episodes,
beta noise 0.3, O = 4, np = 50, nr = 5.  The four cost functions solve the episodes (`solve_batch`: cost_obs, and sigma for mmd_opt);
their plans are validated with counter-based noise (`risk_stats_batch(..., rng="jax")`) at 10^3, 10^4 and 10^5 rollouts.  Each solver
estimate is set against its Monte-Carlo counterpart (DESIGN.md section 3 item 9):

    saa         cost_obs = P(c > 0) from nr rollouts             vs  p_coll
    cvar        cost_obs = CVaR_0.98(c) from nr rollouts          vs  cvar_obs at alpha 0.98
    mmd_opt     cost_obs = weighted reduced-set MMD, sigma        vs  mmd_obs with the plan's sigma
    mmd_random  cost_obs = MMD of nr rollouts, sigma = 0.01       vs  mmd_obs with sigma 0.01

and the mean absolute error and the Spearman rank correlation are recorded per cost function and rollout count.  Wall time of each
synchronous call; device times of the rollout kernel (k_validate_jax<true>) and the statistics kernel (k_risk_stats) from torch.profiler
in a separate call per rollout count; the GPU's name and power limit read in the same run.
usage: risk_probe.py [OUT.json]   (prints the record; also writes it to OUT.json if given)"""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mpc-mmd_b200")):
    sys.path.insert(1, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy.stats import spearmanr  # noqa: E402
import __graft_entry__ as G_  # noqa: E402

G_.build()
from mpcmmd_b200 import CEM, scenes, validation as V  # noqa: E402

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
N_EP, COSTS, ROLLS = 200, ("saa", "cvar", "mmd_opt", "mmd_random"), (1000, 10000, 100000)
MC_KEY = dict(saa="p_coll", cvar="cvar_obs", mmd_opt="mmd_obs", mmd_random="mmd_obs")
out = dict(gpu=gpu, workload="configs[1] sweep point: %d static episodes, beta noise 0.3, O = 4, np = 50, nr = 5; plans of saa, cvar, "
                              "mmd_opt, mmd_random validated with rng=jax at %s rollouts" % (N_EP, list(ROLLS)), pairs=MC_KEY, runs=[])

prob = CEM(5, 4, 0.3, 50, "beta", 0.0, 0.0, variant="static", max_episodes=N_EP)
eps = list(range(N_EP))
batch = scenes.static_batch(prob, eps)
init_state = scenes.driver_inputs("static")[0]
plans = {}
for cost in COSTS:
    sol = prob.solve_batch(cost, **batch)
    items = []
    for k in eps:
        (x, y, vx, vy, _), _ = scenes.static_scene(4, k)
        items.append(dict(cx=sol["cx"][k].astype(np.float64), cy=sol["cy"][k].astype(np.float64), init_state=init_state.astype(np.float64), key=k,
                          x_obs=x.astype(np.float64), y_obs=y.astype(np.float64), vx_obs=vx, vy_obs=vy))
    sigma = np.asarray(sol["sigma"], np.float64) if cost == "mmd_opt" else (np.full(N_EP, 0.01) if cost == "mmd_random" else None)
    plans[cost] = (items, np.asarray(sol["cost_obs"], np.float64), sigma)


def kernel_ms(items, sigma, n_roll):
    """device time of the rollout and statistics kernels of one call, from torch.profiler's CUDA activity records"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        V.risk_stats_batch(prob, items, 50, 0.3, "beta", 4, n_roll=n_roll, rng="jax", sigma=sigma, device=0)
    ms = {}
    for e in prof.key_averages():
        for name in ("k_validate_jax", "k_risk_stats", "k_validate_finish"):
            if name in e.key:
                ms[name] = ms.get(name, 0.0) + e.device_time_total / 1e3
    return ms


all_items = [it for c in COSTS for it in plans[c][0]]
V.risk_stats_batch(prob, all_items[:2], 50, 0.3, "beta", 4, n_roll=1000, rng="jax", device=0)        # warm-up: module load
for n_roll in ROLLS:
    res = dict(n_roll=n_roll, per_cost={})
    for cost in COSTS:
        items, est, sigma = plans[cost]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = V.risk_stats_batch(prob, items, 50, 0.3, "beta", 4, n_roll=n_roll, rng="jax", alpha=0.98, sigma=sigma, device=0)
        wall = time.perf_counter() - t0
        mc = r[MC_KEY[cost]]
        rho = spearmanr(est, mc).correlation if np.ptp(est) > 0 and np.ptp(mc) > 0 else None
        res["per_cost"][cost] = dict(wall_s=wall, mae=float(np.mean(np.abs(est - mc))), spearman=None if rho is None else float(rho),
                                     mean_solver=float(np.mean(est)), mean_mc=float(np.mean(mc)), mean_p_coll=float(np.mean(r["p_coll"])),
                                     plans_with_collisions=int(np.count_nonzero(r["p_coll"] > 0)))
    # all 4 x 200 plans in one call (no MMD, as the CLI runs it): wall time, then the kernels' device times under the profiler
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    V.risk_stats_batch(prob, all_items, 50, 0.3, "beta", 4, n_roll=n_roll, rng="jax", device=0)
    res["all_plans"] = len(all_items)
    res["all_plans_wall_s"] = time.perf_counter() - t0
    res["all_plans_kernel_ms"] = kernel_ms(all_items, None, n_roll)
    k = res["all_plans_kernel_ms"]
    if k.get("k_validate_jax"):
        res["stats_over_rollout_kernel"] = k.get("k_risk_stats", 0.0) / k["k_validate_jax"]
    out["runs"].append(res)
    print(json.dumps(res), flush=True)
if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as f:
        json.dump(out, f, indent=1)
print(json.dumps(out, indent=1))
