#!/usr/bin/env python
"""bench.py -- MPC solves/sec of the B200 trajectory-optimizer path on BASELINE.json's cfg2 workload.

    python bench.py [--gpus N] [--steps K] [--warmup W]                 # this repo's CUDA path
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W] # the CPU baseline arm (oracle port, all host threads)

One "step" = the 200-episode static sweep of synthetic_static_obs/main_mpc.py:106-128 solved with BOTH cost
functions of configs[1] (`cvar` and `mmd_opt`; beta noise 0.3, num_obs 4, num_prime 50, num_reduced 5) = 400 solves.
Multi-GPU is STRONG scaling, the metric BASELINE.json states ("8 GPU, 200-config sweep"): the 200 episodes are sharded
over the ranks exactly as mpcmmd_b200/driver.py::shard does (rank r solves k = r, r + W, ...), no data-path collective; the only
exchange is the NCCL all_gather of the 26-float per-episode record.  `--scaling weak` (200 episodes per GPU) is kept as an option
and its value is reported under `weak_scaling` in the same line.  Prints ONE JSON line on rank 0.

`--dump-outputs DIR` writes what the timed path returned in its last timed step (cx, cy, cost_lane, cost_obs, beta, sigma, res_beta of
every cost function) as DIR/<cost>_<field>.npy.  The inputs are generated from fixed seeds, so two builds run with the same arguments
can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "mpc-mmd_b200")):
    if p not in sys.path:
        sys.path.insert(1, p)
sys.dont_write_bytecode = True         # the benchmark writes nothing into the tree it runs from (which may be read-only)

WORK = dict(num_reduced=5, num_obs=4, noise_level=0.3, num_prime=50, noise="beta", acc_const_noise=0.0, steer_const_noise=0.0)
COSTS = ("cvar", "mmd_opt")
EPISODES = 200
VARIANT = "static"
CEM_KW = {}
WORKLOAD_NAME = ("configs[1]: synthetic_static_obs, cvar + mmd_opt, beta noise 0.3, num_obs 4, num_prime 50, num_reduced 5, "
                 "200-episode sweep (400 solves/step)")
METRIC = "MPC solves/sec"
CONCURRENT_MIN_SAMPLES = 7500          # CEM samples per launch (episodes x num_batch) from which the cost functions of a step solve concurrently on two streams

# The default (and the driver's) workload is configs[1].  The other BASELINE configs are parity-test cases (tests/); `--workload` lets
# them be timed with the same harness for the numbers quoted in DESIGN.md / profiles/ -- those lines are not the headline.
WORKLOADS = {
    "cfg2": dict(work=dict(WORK), costs=COSTS, episodes=EPISODES, variant=VARIANT, kw={}, name=WORKLOAD_NAME),
    "cfg3": dict(work=dict(num_reduced=5, num_obs=6, noise_level=0.1, num_prime=60, noise="gaussian", acc_const_noise=0.0, steer_const_noise=0.0),
                 costs=("mmd_opt",), episodes=200, variant="dynamic", kw={},
                 name="configs[2]: synthetic_dynamic_obs, mmd_opt, gaussian noise 0.1, num_obs 6, num_prime 60, num_reduced 5, 200-episode sweep"),
    "cfg3b": dict(work=dict(num_reduced=5, num_obs=6, noise_level=0.3, num_prime=60, noise="beta", acc_const_noise=0.0, steer_const_noise=0.0),
                  costs=("mmd_opt",), episodes=200, variant="dynamic", kw={},
                  name="configs[2]: synthetic_dynamic_obs, mmd_opt, beta noise 0.3, num_obs 6, num_prime 60, num_reduced 5, 200-episode sweep"),
    "cfg5": dict(work=dict(num_reduced=5, num_obs=32, noise_level=0.1, num_prime=100, noise="gaussian", acc_const_noise=0.0, steer_const_noise=0.0),
                 costs=("cvar",), episodes=25, variant="static", kw=dict(num_batch=16384),
                 name="configs[4] (scaled synthetic): cvar, 16384 CEM samples x 32 obstacles x num_prime 100, 25 episodes per GPU per step "
                      "(the 200-per-GPU sweep is 8 such steps)"),
}


def select_workload(name):
    global WORK, COSTS, EPISODES, VARIANT, CEM_KW, WORKLOAD_NAME
    w = WORKLOADS[name]
    WORK, COSTS, EPISODES, VARIANT, CEM_KW, WORKLOAD_NAME = w["work"], w["costs"], w["episodes"], w["variant"], w["kw"], w["name"]


def cem_args():
    w = WORK
    return (w["num_reduced"], w["num_obs"], w["noise_level"], w["num_prime"], w["noise"], w["acc_const_noise"], w["steer_const_noise"])


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (the reference itself needs jax==0.3.23, absent from this image), naive formulation
def cpu_arm_step(ora, O, episodes):
    """solve `episodes` with both costs on the host; returns number of solves"""
    from mpcmmd_b200 import scenes            # host-only scene generators (NumPy), shared with the CUDA arm so both solve the same inputs
    init_state, mean, cov, v_des = scenes.driver_inputs(VARIANT)
    n = 0
    for k in episodes:
        if VARIANT == "dynamic":
            _, idx, xo, yo = scenes.dynamic_scene(WORK["num_obs"], k)
        else:
            sc, idx = scenes.static_scene(WORK["num_obs"], k) if WORK["num_obs"] <= 9 else scenes.scaled_scene(WORK["num_obs"], k)
            xo, yo, _ = ora.compute_obs_trajectories(*sc)
        for cost in COSTS:
            ora.solve(cost, idx, init_state, mean, cov, xo, yo, v_des)
            n += 1
    return n


def make_cpu_arm():
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    O.set_threads(cores)
    ora = O.OracleCEM(*cem_args(), variant=VARIANT, naive=True, **CEM_KW)
    return ora, O, cores


def line_config(scaling):
    """the `config` object of the JSON line: identical in the native and the reference arm (same workload, same parameters)"""
    return {"workload": WORKLOAD_NAME, "episodes": EPISODES, "costs": list(COSTS), "num_batch": CEM_KW.get("num_batch", 100), "maxiter_cem": 20,
            "sharding": "episode k -> rank k mod W (strong)" if scaling == "strong" else "%d episodes per rank (weak)" % EPISODES}


def run_reference(args, emit):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    ora, O, cores = make_cpu_arm()
    REF_EPISODES = [0, 1, 2, 3]          # bounded sample of the sweep per step (about 3.5 s of CPU work per step on 16 threads)
    sample = "episodes 0-3 of the 200-episode sweep x {%s} = %d solves per step; scalar C port of the reference (oracle, naive formulation), %d host threads" % (
        ", ".join(COSTS), len(COSTS) * len(REF_EPISODES), cores)
    for _ in range(args.warmup):
        cpu_arm_step(ora, O, REF_EPISODES)
    t0 = time.perf_counter()
    n = 0
    for _ in range(args.steps):
        n += cpu_arm_step(ora, O, REF_EPISODES)
    dt = time.perf_counter() - t0
    val = n / dt
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": "solves/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": line_config(args.scaling),
            "cpu_baseline": {"value": val, "unit": "solves/s", "cores": cores, "kind": "port", "sample": sample,
                             "note": "GPU-over-scalar-C-port figure: the reference's own runtime (XLA:CPU under jax==0.3.23) is absent from this image"},
            "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)
    return 0


# ---------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self._stop, self._th = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop.wait(0.05)

    def __enter__(self):
        self._th = threading.Thread(target=self._run, daemon=True); self._th.start(); return self

    def __exit__(self, *a):
        self._stop.set(); self._th.join(timeout=6)

    def summary(self):
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def shard(total, rank, world, scaling):
    """strong: the sweep's episodes k = rank, rank + W, ... (driver.py::shard); weak: `total` episodes of its own per rank"""
    return list(range(rank, total, world)) if scaling == "strong" else list(range(rank * total, rank * total + total))


def traffic_per_launch():
    """dram bytes of one risk-stage launch group of configs[1], from the committed `ncu --set full` capture of this build
    (profiles/r02_traffic.json, written by tools/ncu_traffic.py from the raw CSV export); None when no capture of this build is committed"""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        return float(t["dram_bytes_per_risk_launch"]), t.get("source")
    except Exception:
        return None, None


DUMP_CAP_BYTES = 64 << 20


def write_outputs(out_dir, arrays, cap=DUMP_CAP_BYTES):
    """--dump-outputs: each array (one row per episode, the same rows in all) as out_dir/<name>.npy in float32.  Above `cap` bytes in all,
    every array keeps the same seeded sample of rows and the kept row indices go to out_dir/rows.npy (float64)."""
    arrays = {k: np.ascontiguousarray(v, dtype=np.float32) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    if total > cap:
        n = next(iter(arrays.values())).shape[0]
        rows = np.sort(np.random.default_rng(0).choice(n, int(cap // (total / n + 8)), replace=False))
        arrays = {k: a[rows] for k, a in arrays.items()}
        arrays["rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)
    return sorted(arrays)


def main():
    # The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout), so everything
    # except the final line is routed to stderr: fd 1 is pointed at fd 2 for the run and the line goes to the saved descriptor.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(real_stdout, (json.dumps(line) + "\n").encode())

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"],
                    help="strong (default, BASELINE's metric): the 200-episode sweep sharded over the ranks; weak: 200 episodes per rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other BASELINE workloads / the weak-scaling value / the batch-1 latency")
    ap.add_argument("--episodes", type=int, default=0, help="diagnostic: episodes of the sweep (default: the workload's 200); e.g. 25 = one rank's shard of the 8-GPU run")
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--projection", default="exact", choices=["exact", "tc"],
                    help="exact = k_project (bit-exact FP32, the default product path); tc = k_project_tc (tcgen05 kind::tf32 products, 1e-4 stage parity)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the solver returned in the last one as DIR/<cost>_<field>.npy (float32; row i = "
                         "episode i of the sweep; with several ranks DIR/rank<r>/, row i = the rank's i-th episode)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs writes the outputs of the native (CUDA) path")
    if args.projection == "tc":
        os.environ["MPCMMD_PROJ"] = "tc"          # read by mpcmmd_create
    else:
        os.environ.pop("MPCMMD_PROJ", None)
    select_workload(args.workload)
    if args.episodes > 0:
        global EPISODES
        EPISODES = args.episodes
    if args.impl == "reference":
        return run_reference(args, emit)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    import __graft_entry__ as G
    if local == 0:
        G.build()                      # one builder per node; the other ranks wait, then only load
    if world > 1:
        dist.barrier()
    if local != 0:
        G.build()
    from mpcmmd_b200 import CEM, cem_impl, scenes
    W, K = max(args.warmup, 3), args.steps
    keys = ("idx_mpc", "init_state", "mean_param", "cov_param", "x_obs_traj", "y_obs_traj", "v_des")
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)       # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        t = torch.tensor([x], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    class Arm:
        """one workload on this rank's shard: handle, device-resident and pinned-host inputs, the two step flavours"""

        def __init__(self, scaling):
            self.eps = shard(EPISODES, rank, world, scaling)
            self.E = len(self.eps)
            # one handle and one CUDA stream per cost function: the solves of the sweep's cost functions are independent and run concurrently
            # (the reference's main_mpc.py loops over them serially, main_mpc.py:84-104)
            self.probs = {c: CEM(*cem_args(), variant=VARIANT, max_episodes=max(self.E, 1), device=local, **CEM_KW) for c in COSTS}
            self.prob = self.probs[COSTS[-1]]
            self.streams = {c: torch.cuda.Stream(dev) for c in COSTS}
            self.pool = ThreadPoolExecutor(max_workers=len(COSTS))
            # ... when every launch fills the device.  A shard of a few waves of chains (25 / 50 episodes per rank: the 8- / 4-GPU sweep) gains nothing from two
            # concurrent graphs -- the short latency-bound kernels of cvar and the chain waves of mmd_opt only delay each other (tools/overlap_probe.py: 25 episodes
            # 24.8 ms concurrent, 24.4 ms back to back; 50: 45.8 / 44.6; 100: 84.9 / 86.7) -- so small shards solve their cost functions back to back on one stream
            self.concurrent = len(COSTS) > 1 and self.E * self.probs[COSTS[0]].num_batch >= CONCURRENT_MIN_SAMPLES
            self.host = scenes.static_batch(self.prob, self.eps, VARIANT)
            self.dev_in = {k: torch.as_tensor(self.host[k], device=dev) for k in keys}
            self.pinned_np = {k: torch.as_tensor(self.host[k]).pin_memory().numpy() for k in keys}
            self.thresholds = {c: (-self.prob.ker_wt + 1.0 if c in ("mmd_opt", "mmd_random") else 1e-5) for c in COSTS}     # main_mpc.py:88-97
            self.k_col = torch.as_tensor(self.eps, device=dev, dtype=torch.float32)[:, None]
            self.total_solves = EPISODES * len(COSTS) * (1 if scaling == "strong" else world)

        def record(self, outs):
            """26-float per-episode records [k, accepted, cost_obs, cost_lane, cx(11), cy(11)] of every cost function, gathered over the ranks in ONE
            NCCL all_gather (SURVEY 8e).  Shards are ragged under strong scaling (200 = 8 x 25 is even, 3- or 7-way is not): every rank pads to the
            largest shard with k = -1 rows, which `unpad` drops after the timed region (boolean indexing would synchronise the host inside it)."""
            recs = []
            for cost in COSTS:
                out = outs[cost]
                recs.append(torch.cat([self.k_col, (out["cost_obs"] <= self.thresholds[cost]).float()[:, None], out["cost_obs"][:, None],
                                       out["cost_lane"][:, None], out["cx"], out["cy"]], 1))
            rec = torch.stack(recs, 0)                                  # (costs, E, 26)
            if world > 1:
                m = (EPISODES + world - 1) // world if len(self.eps) != EPISODES else EPISODES
                pad = torch.full((len(COSTS), m, 26), -1.0, device=dev); pad[:, :rec.shape[1]] = rec
                buf = torch.empty((world,) + tuple(pad.shape), device=dev)
                dist.all_gather_into_tensor(buf, pad)
                rec = buf.permute(1, 0, 2, 3).reshape(len(COSTS), world * m, 26)
            return rec

        @staticmethod
        def unpad(rec):
            return {cost: rec[i][rec[i][:, 0] >= 0] for i, cost in enumerate(COSTS)}

        def step_device(self):
            cur = torch.cuda.current_stream(dev)
            outs = {}
            self.last_outs = outs                                       # what the solver handed back in this step (--dump-outputs)
            if not self.concurrent:
                for cost in COSTS:
                    outs[cost] = self.probs[cost].solve_batch_device(cost, *[self.dev_in[k] for k in keys])
                return self.record(outs)
            for cost in COSTS:
                st = self.streams[cost]
                st.wait_stream(cur)
                with torch.cuda.stream(st):
                    outs[cost] = self.probs[cost].solve_batch_device(cost, *[self.dev_in[k] for k in keys])
            for cost in COSTS:
                cur.wait_stream(self.streams[cost])
            return self.record(outs)

        def step_host(self):
            """host buffers in, host buffers out: one synchronous C-ABI call per cost function, issued from one host thread each"""
            if not self.concurrent:
                return {cost: self.probs[cost].solve_batch(cost, *[self.pinned_np[k] for k in keys]) for cost in COSTS}
            futs = {cost: self.pool.submit(self.probs[cost].solve_batch, cost, *[self.pinned_np[k] for k in keys]) for cost in COSTS}
            return {cost: f.result() for cost, f in futs.items()}

        def time_device(self, K, W, clocks=None):
            """K timed steps, device-resident inputs, CUDA events per step, L2 flushed between steps; returns (ms_total max over ranks, wall, recs, launches/step)"""
            for _ in range(W):
                self.step_device()
            launches = 0
            for cost in COSTS:            # graphs are cached now; count launches per solve batch
                self.probs[cost].solve_batch_device(cost, *[self.dev_in[k] for k in keys]); launches += self.probs[cost].last_launch_count()
            barrier()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
            barrier()
            t0 = time.perf_counter()
            for i in range(K):
                flush.fill_(i & 0xFF)                       # L2 flush between timed steps (outside the event pair)
                ev[i][0].record()
                recs = self.step_device()
                ev[i][1].record()
            barrier()
            wall = time.perf_counter() - t0
            self.step_ms = [a.elapsed_time(b) for a, b in ev]
            return max_over_ranks(sum(self.step_ms)), wall, self.unpad(recs), launches

    def _time_median(self):
        """extra keys only: median of 3 timed steps after 3 warm-up steps (max over ranks), robust against a one-off slow step"""
        _, _, recs, _ = self.time_device(3, 3)
        self.last_recs = recs
        return max_over_ranks(float(np.median(self.step_ms)))
    Arm.time_median = _time_median

    # ---- device-resident throughput (`value`) on the headline workload
    arm = Arm(args.scaling)
    prob, E = arm.prob, arm.E
    concurrent_flag = arm.concurrent
    HEAVY = COSTS[-1]                                                             # the cost whose risk stage the roofline describes
    with ClockSampler(local) as clk:
        ms_total, t_wall, recs, launches_per_step = arm.time_device(K, W)
    value = arm.total_solves * K / (ms_total * 1e-3)
    accepted = {c: int(recs[c][:, 1].sum().item()) for c in COSTS}
    if args.dump_outputs:
        write_outputs(args.dump_outputs if world == 1 else os.path.join(args.dump_outputs, "rank%d" % rank),
                      {"%s_%s" % (c, f): v.cpu().numpy() for c, o in arm.last_outs.items() for f, v in o.items() if not f.startswith("_")})

    # ---- end to end through the host-buffer C ABI call (`e2e`): pinned host inputs, H2D + D2H inside the timed region
    for _ in range(2):
        arm.step_host()
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        outs = arm.step_host()
    barrier()
    e2e_value = arm.total_solves * K / max_over_ranks(time.perf_counter() - t0)
    h2d = len(COSTS) * sum(int(arm.pinned_np[k].nbytes) for k in keys)
    d2h = len(COSTS) * sum(int(v.nbytes) for v in outs[HEAVY].values())
    mine = {c: recs[c][torch.isin(recs[c][:, 0], torch.as_tensor(arm.eps, device=dev, dtype=torch.float32))] for c in COSTS}     # this rank's rows of the gathered records
    same = all(np.array_equal(outs[c]["cx"], mine[c][torch.argsort(mine[c][:, 0])][:, 4:15].cpu().numpy()) for c in COSTS)        # arm.eps ascends

    # ---- roofline of the dominant kernel group (risk stage of the heavy cost), launch-by-launch CUDA events on the launching stream
    prob.solve_batch_device(HEAVY, *[arm.dev_in[k] for k in keys]); torch.cuda.synchronize()
    prof = prob.profile_solve(HEAVY, E)
    prof_cvar = None
    if "cvar" in COSTS and HEAVY != "cvar":
        arm.probs["cvar"].solve_batch_device("cvar", *[arm.dev_in[k] for k in keys]); torch.cuda.synchronize()
        prof_cvar = arm.probs["cvar"].profile_solve("cvar", E)
    fl = scenes.flops_per_sample(HEAVY, WORK["num_reduced"], WORK["num_prime"], WORK["num_obs"])
    flops_per_launch = fl["risk"] * prob.num_batch * E
    avg_launch_s = prof["ms"]["risk"] * 1e-3 / prof["launches"]["risk"]
    peak_tf, sm_count = cem_impl.fp32_peak(local)
    achieved = flops_per_launch / avg_launch_s / 1e12
    traffic, traffic_src = traffic_per_launch() if (args.workload == "cfg2" and world == 1) else (None, None)
    roofline = {"bound": "fp32", "kernel": ("risk stage of mmd_opt: k_rollouts<ROLL_OPT> + reduced-set inner CEM (%s) + k_opt_risk" % prob.inner_cem_path() if HEAVY == "mmd_opt"
                                            else "k_rollouts (noisy rollouts + %s risk)" % HEAVY), "achieved": achieved, "peak": peak_tf,
                "unit": "TFLOP/s", "frac": achieved / peak_tf, "traffic": traffic, "traffic_source": traffic_src,
                "peak_source": "measured in this run: register-resident FP32 fma micro-kernel (MEASURED_PEAKS.json has no FP32 figure)",
                "flops_per_launch": flops_per_launch, "avg_launch_ms": avg_launch_s * 1e3, "sm_count": sm_count, "episodes_per_launch": E,
                "xu_peaks_measured": cem_impl.xu_peaks(local),
                "kernel_share_of_%s_solve" % HEAVY: prof["ms"]["risk"] / prof["ms"]["total"],
                "%s_ms_by_kernel" % HEAVY: prof["ms"]}
    if prof_cvar:
        roofline["cvar_ms_by_kernel"] = prof_cvar["ms"]

    # ---- per-solve latency at batch = 1 (BASELINE.json's second headline)
    lat = {}
    if rank == 0 and not args.no_extras:
        p1 = CEM(*cem_args(), variant=VARIANT, max_episodes=1, device=local, **CEM_KW)
        one = {k: arm.dev_in[k][:1].contiguous() for k in keys}
        host = arm.host
        for cost in COSTS:
            for _ in range(5):
                p1.solve_batch_device(cost, *[one[k] for k in keys])
            torch.cuda.synchronize()
            ts = []
            for _ in range(30):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record(); p1.solve_batch_device(cost, *[one[k] for k in keys]); b.record(); torch.cuda.synchronize()
                ts.append(a.elapsed_time(b))
            # the same solve through the reference-facing call (CEM.compute_cem_*: host arrays in, host arrays out, wall clock)
            fn = getattr(p1, "compute_cem_" + cost)
            h1 = [int(host["idx_mpc"][0]), host["init_state"][0], host["mean_param"][0], host["cov_param"][0], host["x_obs_traj"][0], host["y_obs_traj"][0],
                  float(host["v_des"][0])]
            for _ in range(5):
                fn(*h1)
            tw = []
            for _ in range(30):
                t0 = time.perf_counter(); fn(*h1); tw.append(1e3 * (time.perf_counter() - t0))
            lat[cost] = {"p50_ms": float(np.percentile(ts, 50)), "p95_ms": float(np.percentile(ts, 95)),
                         "p50_ms_host_api": float(np.percentile(tw, 50)), "p95_ms_host_api": float(np.percentile(tw, 95)),
                         "ms_by_kernel_ungraphed": p1.profile_solve(cost, 1)["ms"]}
        del p1
    del arm, prob
    torch.cuda.empty_cache()

    # ---- the other BASELINE workloads and the weak-scaled value, device-resident, same timing rules (extra keys; not the headline)
    extras, weak, modes = {}, None, {}
    if not args.no_extras and args.workload == "cfg2":
        if args.scaling == "strong" and world > 1:
            a2 = Arm("weak")
            ms2 = a2.time_median()
            weak = {"value": a2.total_solves / (ms2 * 1e-3), "unit": "solves/s", "episodes_per_gpu": EPISODES, "ms_per_step": ms2}
            del a2
            torch.cuda.empty_cache()
        for name, scal in (("cfg3", args.scaling), ("cfg3b", args.scaling), ("cfg5", "weak")):
            select_workload(name)
            a3 = Arm(scal)
            ms3 = a3.time_median(); r3 = a3.last_recs
            extras[name] = {"workload": WORKLOAD_NAME, "value": a3.total_solves / (ms3 * 1e-3), "unit": "solves/s", "ms_per_step": ms3,
                            "scaling": scal, "episodes_this_rank": a3.E, "step_ms": a3.step_ms, "accepted": {c: int(r3[c][:, 1].sum().item()) for c in COSTS}}
            del a3
            torch.cuda.empty_cache()
        select_workload(args.workload)
        # opt-in modes on the headline workload (tolerance parity, never the default): tensor-core projection and MUFU exponentials
        for name, env, wl in (("projection_tc", {"MPCMMD_PROJ": "tc"}, None), ("fast_math", {"MPCMMD_MATH": "fast"}, None),
                              ("cfg5_projection_tc", {"MPCMMD_PROJ": "tc"}, "cfg5")):      # the scaled configuration is where the projection weighs most (44 % of its step)
            if args.projection == "tc" and env.get("MPCMMD_PROJ") == "tc":
                continue
            os.environ.update(env)
            if wl:
                select_workload(wl)
            a4 = Arm("weak" if wl == "cfg5" else args.scaling)
            ms4 = a4.time_median(); r4 = a4.last_recs
            modes[name] = {"env": env, "workload": WORKLOAD_NAME, "value": a4.total_solves / (ms4 * 1e-3), "unit": "solves/s", "ms_per_step": ms4,
                           "accepted": {c: int(r4[c][:, 1].sum().item()) for c in COSTS},
                           "parity": "stage outputs within 1e-4 of the reference fixtures (tests); not bit-exact, not the default"}
            for k in env:
                os.environ.pop(k, None)
            del a4
            torch.cuda.empty_cache()
            if wl:
                select_workload(args.workload)

    # ---- CPU baseline beside it (rank 0, N = 1 only): bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        ora, O, cores = make_cpu_arm()
        t0 = time.perf_counter()
        n = cpu_arm_step(ora, O, list(range(12)))
        dt = time.perf_counter() - t0
        cpu = {"value": n / dt, "unit": "solves/s", "cores": cores, "kind": "port",
               "sample": "episodes 0-11 of the sweep x {%s} = %d solves in %.1f s; oracle port (scalar C, reference's naive formulation; NOT XLA:CPU), %d host threads" % (", ".join(COSTS), n, dt, cores)}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "solves/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_total / K,
                "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                "config": line_config(args.scaling),
                "details": {"episodes_this_rank": E, "projection": args.projection, "concurrency": ("one handle + CUDA stream per cost function (cvar and mmd_opt solve concurrently)" if concurrent_flag else "one handle per cost function, solved back to back on one stream (shard too small for concurrent graphs to pay)"), "l2": "flushed between timed steps (256 MiB fill)",
                            "parallelism": "episodes sharded %d-way, no data-path collective" % world, "accepted": accepted, "wall_s_timed_region": t_wall},
                "e2e": {"value": e2e_value, "unit": "solves/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "matches_device_path": bool(same)},
                "gpu_launches": launches_per_step * K, "roofline": roofline, "cpu_baseline": cpu, "latency_1gpu_batch1": lat,
                "other_workloads": extras, "opt_in_modes": modes, "weak_scaling": weak, "clocks": clk.summary()}
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
