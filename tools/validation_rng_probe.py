#!/usr/bin/env python
"""Monte-Carlo validation of one configs[1] sweep point in its three noise modes: the legacy-stream noise drawn on the host (NumPy, the
default) and on the device (`compute_stats_batch(..., rng="device")`), and counter-based JAX-protocol noise drawn by the rollout kernel
(`rng="jax"`).  200 static episodes solved with cvar and mmd_opt (beta noise 0.3, O = 4, np = 50, nr = 5), the scenes both solved
validated with both costs, 1000 rollouts each -- what `validation.py` runs per sweep point.  Repeated with Gaussian noise 0.3.  Each path
is warmed up once on two trajectories, then timed on all of them; a wall clock that ends when the synchronous call returns.  The counts
of the two legacy-stream paths are compared.  The JAX mode is also timed at 10^5 rollouts per trajectory (the legacy-stream modes cost
about 100x their 1000-rollout time there and are not run).  One extra call per (mode, rollout count) under torch.profiler gives the
kernels' device times.  usage: validation_rng_probe.py [OUT.json]   (prints the record; also writes it to OUT.json if given)"""
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mpc-mmd_b200")):
    sys.path.insert(1, p)
import numpy as np  # noqa: E402
import torch  # noqa: E402
import __graft_entry__ as G_  # noqa: E402

G_.build()
from mpcmmd_b200 import CEM, driver, validation as V  # noqa: E402

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"], capture_output=True,
                     text=True).stdout.strip()
out = dict(gpu=gpu, workload="configs[1] sweep point: 200 static episodes, cvar + mmd_opt, O = 4, np = 50, nr = 5, 1000 rollouts per trajectory "
                             "(and 10^5 for rng=jax)", runs=[])


def kernel_ms(**kw):
    """device time of the k_validate* kernels of one call, from torch.profiler's CUDA activity records"""
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        V.compute_stats_batch(prob, items, 50, 0.3, noise, 4, **kw)
    return {e.key: e.device_time_total / 1e3 for e in prof.key_averages() if e.key.startswith("k_validate")}



tmp = tempfile.mkdtemp(prefix="validation_rng_probe_")
for noise in ("beta", "gaussian"):
    common = ["--noises", noise, "--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "4", "--num_prime", "50",
              "--acc_const_noise", "0.0", "--steer_const_noise", "0.0", "--root", os.path.join(tmp, "data")]
    driver.run_sweep(driver.build_parser().parse_args(common + ["--costs", "cvar", "mmd_opt", "--num_configs", "200"]), log=lambda *a: None)
    d_o = V._load(os.path.join(tmp, "data"), noise, 0.3, 50, "mmd_opt", 5, 4)
    d_c = V._load(os.path.join(tmp, "data"), noise, 0.3, 50, "cvar", 5, 4)
    pairs = V.matched_pairs(d_c, d_o, 4)
    items = [V._item(d_o, im, k, False) for k, _, im in pairs] + [V._item(d_c, ic, k, False) for k, ic, _ in pairs]
    prob = CEM(5, 4, 0.3, 50, noise, 0.0, 0.0, variant="static", max_episodes=1)
    res = dict(noise=noise, noise_level=0.3, trajectories=len(items))
    for rng in ("host", "device", "jax"):
        V.compute_stats_batch(prob, items[:2], 50, 0.3, noise, 4, rng=rng)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res[rng] = V.compute_stats_batch(prob, items, 50, 0.3, noise, 4, rng=rng)
        res[rng + "_s"] = time.perf_counter() - t0
    for rng in ("device", "jax"):
        res[rng + "_s_repeats"] = []
        for _ in range(3):
            t0 = time.perf_counter()
            V.compute_stats_batch(prob, items, 50, 0.3, noise, 4, rng=rng)
            res[rng + "_s_repeats"].append(time.perf_counter() - t0)
    res["counts_equal"] = bool(np.array_equal(res["host"][0], res["device"][0]) and np.array_equal(res["host"][1], res["device"][1]))
    # the JAX mode draws other numbers from the same distributions: its mean collision / lane fractions next to NumPy's
    res["mean_count_fraction"] = {rng: [float(np.mean(res[rng][0])) / 1000, float(np.mean(res[rng][1])) / 1000] for rng in ("host", "jax")}
    del res["host"], res["device"], res["jax"]
    res["ratio_host_over_device"] = res["host_s"] / res["device_s"]
    res["ratio_device_over_jax"] = min(res["device_s_repeats"]) / min(res["jax_s_repeats"])
    res["kernel_ms"] = kernel_ms(rng="device")
    res["jax_kernel_ms"] = kernel_ms(rng="jax")
    n5 = 100000
    V.compute_stats_batch(prob, items[:2], 50, 0.3, noise, 4, rng="jax", n_roll=n5)
    res["jax_1e5_s_repeats"] = []
    for _ in range(3):
        t0 = time.perf_counter()
        c5 = V.compute_stats_batch(prob, items, 50, 0.3, noise, 4, rng="jax", n_roll=n5)
        res["jax_1e5_s_repeats"].append(time.perf_counter() - t0)
    res["jax_1e5_mean_count_fraction"] = [float(np.mean(c5[0])) / n5, float(np.mean(c5[1])) / n5]
    res["jax_1e5_kernel_ms"] = kernel_ms(rng="jax", n_roll=n5)
    out["runs"].append(res)
    print(json.dumps(res), flush=True)
    del prob
shutil.rmtree(tmp)
if len(sys.argv) > 1:
    os.makedirs(os.path.dirname(os.path.abspath(sys.argv[1])), exist_ok=True)
    with open(sys.argv[1], "w") as f:
        json.dump(out, f, indent=1)
print(json.dumps(out, indent=1))
