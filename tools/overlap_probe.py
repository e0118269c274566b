#!/usr/bin/env python
"""Strong-scaled shard of the sweep on ONE GPU (E = 25 / 50 / 100 episodes = the per-rank share at 8 / 4 / 2 GPUs): the cvar + mmd_opt step of bench.py
(one handle + stream per cost function, concurrent) for each number of episode groups (branches) of the mmd_opt solve graph (MPCMMD_GROUPS).
usage: [PROBE_GROUPS=1,2,3,4] overlap_probe.py [E ...]      (writes overlap_probe.json to the output directory at the end of the script)"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "mpc-mmd_b200")):
    sys.path.insert(1, p)
import torch  # noqa: E402
import __graft_entry__ as G_  # noqa: E402

G_.build()
from mpcmmd_b200 import CEM, scenes  # noqa: E402

args = (5, 4, 0.3, 50, "beta", 0.0, 0.0)
keys = ("idx_mpc", "init_state", "mean_param", "cov_param", "x_obs_traj", "y_obs_traj", "v_des")
dev = torch.device("cuda", 0)
flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)


def timed(fn, n=9):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for i in range(n):
        flush.fill_(i)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


out = {}
Es = [int(a) for a in sys.argv[1:]] or [25, 50, 100]
GROUPS = os.environ.get("PROBE_GROUPS", "1,2,3,4").split(",")
for E in Es:
    host = None
    for groups in GROUPS:
        hs = {}
        for c in ("cvar", "mmd_opt"):
            os.environ["MPCMMD_GROUPS"] = groups if c == "mmd_opt" else "1"
            hs[c] = CEM(*args, variant="static", max_episodes=E, device=0)
        if host is None:
            host = scenes.static_batch(hs["cvar"], list(range(E)), "static")
            dev_in = {k: torch.as_tensor(host[k], device=dev) for k in keys}
        streams = {c: torch.cuda.Stream(dev) for c in hs}

        def serial():
            for c in ("cvar", "mmd_opt"):
                hs[c].solve_batch_device(c, *[dev_in[k] for k in keys])

        def step(which=("cvar", "mmd_opt")):
            cur = torch.cuda.current_stream(dev)
            for c in which:
                streams[c].wait_stream(cur)
                with torch.cuda.stream(streams[c]):
                    hs[c].solve_batch_device(c, *[dev_in[k] for k in keys])
            for c in which:
                cur.wait_stream(streams[c])
        t_both = timed(step)
        t_opt = timed(lambda: step(("mmd_opt",)))
        t_cvar = timed(lambda: step(("cvar",)))
        tag = "E%d_g%s" % (E, groups)
        t_serial = timed(serial)
        out[tag] = {"both_ms": t_both, "mmd_opt_ms": t_opt, "cvar_ms": t_cvar, "serial_ms": t_serial}
        print(tag, "both %.3f  mmd_opt %.3f  cvar %.3f  serial (one stream) %.3f" % (t_both, t_opt, t_cvar, t_serial), flush=True)
        del hs
        torch.cuda.empty_cache()
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
json.dump(out, open(os.path.join(ROOT, "gpurun_out", "overlap_probe.json"), "w"), indent=1)
