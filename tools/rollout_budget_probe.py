#!/usr/bin/env python
"""How many rollouts per CEM sample do cvar and saa need?  One configs[1] sweep point: 200 static episodes, beta noise 0.3, O = 4, np = 50.

cvar and saa solve the 200 episodes at num_reduced 5, 25, 64, 100, 256 and 1024 (above 64: k_rollouts_wide); mmd_opt at num_reduced 5 and 8
(25 and 64 mother rollouts per sample) is the comparison.  For every set of plans:
  solve_ms        the 200-episode solve (solve_batch, host arrays, synchronous), warmed, median of REPS calls, host clock;
  p50_batch1_ms   the median of REPS1 one-episode solves, host clock;
  accepted        episodes whose cost_obs passes the driver's threshold (main_mpc.py:86-97: 1e-5 for cvar / saa, 1 - ker_wt for mmd_opt);
  Monte-Carlo risk of the plans from risk_stats_batch(rng="jax", n_roll=10^4): mean p_coll and cvar_obs (alpha 0.98), and the solver's own
  estimate against its Monte-Carlo counterpart (saa: p_coll, cvar: cvar_obs, mmd_opt: mmd_obs with the plan's sigma) as mean absolute error
  and Spearman rank correlation, as tools/risk_probe.py does.
The GPU's name, power limit and max SM clock are read in the same run.
usage: rollout_budget_probe.py [OUT.json]   (prints the record; also writes it to OUT.json if given)"""
import gc
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
from mpcmmd_b200 import CEM, driver, scenes, validation as V  # noqa: E402

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
N_EP, N_ROLL, REPS, REPS1 = 200, 10 ** 4, 5, 21
RUNS = [(c, nr) for c in ("cvar", "saa") for nr in (5, 25, 64, 100, 256, 1024)] + [("mmd_opt", 5), ("mmd_opt", 8)]
MC_KEY = dict(saa="p_coll", cvar="cvar_obs", mmd_opt="mmd_obs")
out = dict(gpu=gpu, workload="configs[1] sweep point: %d static episodes, beta noise 0.3, O = 4, np = 50; Monte-Carlo risk with rng=jax at "
                              "%d rollouts per plan" % (N_EP, N_ROLL), pairs=MC_KEY, runs=[])
eps = list(range(N_EP))
init_state = scenes.driver_inputs("static")[0]


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 3) for t in ts]


for cost, nr in RUNS:
    prob = CEM(nr, 4, 0.3, 50, "beta", 0.0, 0.0, variant="static", max_episodes=N_EP)
    batch = scenes.static_batch(prob, eps)
    one = {k: v[:1] for k, v in batch.items()}
    sol = prob.solve_batch(cost, **batch)                                   # warm-up: graph capture of the 200-episode solve
    prob.solve_batch(cost, **one)                                           # and of the one-episode solve
    solve_ms, solve_all = timed(lambda: prob.solve_batch(cost, **batch), REPS)
    p50_1, _ = timed(lambda: prob.solve_batch(cost, **one), REPS1)
    _, thr = driver.thresholds(prob, cost)
    est = np.asarray(sol["cost_obs"], np.float64)
    items = []
    for k in eps:
        (x, y, vx, vy, _), _ = scenes.static_scene(4, k)
        items.append(dict(cx=sol["cx"][k].astype(np.float64), cy=sol["cy"][k].astype(np.float64), init_state=init_state.astype(np.float64), key=k,
                          x_obs=x.astype(np.float64), y_obs=y.astype(np.float64), vx_obs=vx, vy_obs=vy))
    sigma = np.asarray(sol["sigma"], np.float64) if cost == "mmd_opt" else None
    r = V.risk_stats_batch(prob, items, 50, 0.3, "beta", 4, n_roll=N_ROLL, rng="jax", alpha=0.98, sigma=sigma, device=0)
    mc = np.asarray(r[MC_KEY[cost]], np.float64)
    rho = spearmanr(est, mc).correlation if np.ptp(est) > 0 and np.ptp(mc) > 0 else None
    rec = dict(cost=cost, num_reduced=nr, rollouts_per_sample=nr * nr if cost == "mmd_opt" else nr, solve_ms=solve_ms, solve_ms_all=solve_all,
               p50_batch1_ms=p50_1, accepted=int(np.count_nonzero(est <= thr)), threshold=thr,
               mean_p_coll=float(np.mean(r["p_coll"])), mean_cvar_obs=float(np.mean(r["cvar_obs"])),
               plans_with_collisions=int(np.count_nonzero(np.asarray(r["p_coll"]) > 0)),
               mean_solver=float(np.mean(est)), mean_mc=float(np.mean(mc)), mae=float(np.mean(np.abs(est - mc))),
               spearman=None if rho is None or not np.isfinite(rho) else float(rho))
    out["runs"].append(rec)
    print(json.dumps(rec), flush=True)
    del prob, sol
    gc.collect()
    torch.cuda.empty_cache()
if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as f:
        json.dump(out, f, indent=1)
print(json.dumps(out, indent=1))
