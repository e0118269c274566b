"""BASELINE configs[3] for mmd_opt: one solve (and a batch of 8) per num_reduced in {5, 10, 20, 40} at num_prime 60, 6 obstacles, gaussian noise 0.1.
Large reduced sets run a reduced number of OUTER iterations (every outer iteration costs the same) and are scaled to the reference's 20; the
inner CEM always runs its full 20 iterations x 100 samples.  Prints a markdown table.  Usage: python tools/bench_mmd_opt_nr.py"""
import sys
sys.path.insert(1, "/root/repo"); sys.path.insert(1, "/root/repo/mpc-mmd_b200")
import numpy as np, torch
import __graft_entry__ as G
G.build()
from mpcmmd_b200 import CEM, scenes
keys = ("idx_mpc", "init_state", "mean_param", "cov_param", "x_obs_traj", "y_obs_traj", "v_des")
print("| num_reduced | d = nr^2+1 | episodes | outer iterations timed | ms per solve (scaled to 20 outer iterations) | algorithmic GFLOP per solve | TFLOP/s | kernel path |"); print("|---|---|---|---|---|---|---|---|")
for nr, iters in ((5, 20), (10, 20), (20, 4), (40, 1)):
    for E in (1, 8):
        if nr == 40 and E == 8:
            continue
        prob = CEM(nr, 6, 0.1, 60, "gaussian", 0.0, 0.0, max_episodes=E, maxiter_cem=iters)
        host = scenes.static_batch(prob, list(range(E)), "static")
        dev_in = {k: torch.as_tensor(host[k], device="cuda:0") for k in keys}
        run = lambda: prob.solve_batch_device("mmd_opt", *[dev_in[k] for k in keys])
        run(); torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); run(); b.record(); torch.cuda.synchronize(); ts.append(a.elapsed_time(b))
        ms = float(np.median(ts)) * 20.0 / iters / E
        fl = scenes.flops_per_sample("mmd_opt", nr, 60, 6); gf = (fl["project"] + fl["risk"]) * 100 * 20 / 1e9
        print(f"| {nr} | {nr * nr + 1} | {E} | {iters} | {ms:.1f} | {gf:.1f} | {gf / ms:.2f} | {prob.inner_cem_path()} |", flush=True)
        del prob
