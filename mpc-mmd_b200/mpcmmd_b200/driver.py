"""Sweep driver: the reference's `synthetic_static_obs/main_mpc.py` and `synthetic_dynamic_obs/main_mpc.py` workflows on the
batched B200 solver (`--variant static|dynamic`; the two drop-in `main_mpc.py` files fix it).

Same command line, same loop nest (`noises x noise_levels x num_prime x num_obs x num_reduced_sets x costs`,
main_mpc.py:77-104), same scenes (`compute_obs_data`, :10-21), same per-episode `idx_mpc` draw (:113-119), same
acceptance thresholds (:86-97) and the same on-disk schema (:130-135):

    ./data/{noise}_noise/noise_{int(100*level)}/ts_{num_prime}/{cost}_{num_reduced}_samples_{num_obs}_obs.npz
        cx, cy (n_acc, 11); init_state (n_acc, 6); x_obs, y_obs, vx_obs, vy_obs (n_acc, num_obs)      -- float64, accepted episodes only
        dynamic variant adds psi_obs (n_acc, num_obs), x_obs_traj, y_obs_traj (n_acc, num_obs, 100)      (D/main_mpc.py:150-156)

What differs from the reference: the 200 episodes of a sweep point are solved in ONE `solve_batch` call (they are
independent: every input depends only on (k, num_obs)), optionally sharded over ranks (`episodes k = rank, rank+W, ...`;
the per-episode records are gathered and written by rank 0 in episode order, SURVEY.md section 8e).

`--kernel gaussian` (default `laplace`, the reference's) plans mmd_opt / mmd_random with the Gaussian-kernel MMD; their files then
also hold `kernel="gaussian"`.  The cvar / saa files do not depend on the kernel and are written as always.

    python -m mpcmmd_b200.driver --costs mmd_opt cvar --noises beta --noise_levels 0.3 --num_reduced_sets 5 \\
        --num_obs 4 --num_prime 50 --acc_const_noise 0.0 --steer_const_noise 0.0 [--num_configs 200] [--root ./data]
"""
from __future__ import annotations

import argparse
import os
import time

import numpy as np

from . import scenes
from .cem_impl import CEM

F32 = np.float32
COST_FUNCS = {"mmd_opt": "mmd_opt", "mmd_random": "mmd_random", "cvar": "cvar", "saa": "saa"}


def thresholds(prob, cost):
    """(threshold_lane, threshold_obs) of main_mpc.py:86-97; any cost other than the two MMD ones takes the cvar branch"""
    if cost in ("mmd_opt", "mmd_random"):
        return -2 * prob.ker_wt + 1.0, -prob.ker_wt + 1.0
    return 10 ** (-5), 10 ** (-5)


def solve_cost(cost):
    """main_mpc.py:86-97: mmd_opt / mmd_random have their own entry points, everything else runs compute_cem_cvar"""
    return cost if cost in ("mmd_opt", "mmd_random") else "cvar"


def shard(num_configs: int, rank: int, world: int):
    """episodes of this rank: k = rank, rank + world, ... (SURVEY.md section 8e)"""
    return list(range(rank, num_configs, world))


def pack_records(episodes, out):
    """one 26-float record per episode: [k, cost_obs, cost_lane, cx(11), cy(11), pad]"""
    E = len(episodes)
    rec = np.zeros((E, 26), F32)
    rec[:, 0] = np.asarray(episodes, F32)
    rec[:, 1] = out["cost_obs"]; rec[:, 2] = out["cost_lane"]
    rec[:, 3:14] = out["cx"]; rec[:, 14:25] = out["cy"]
    return rec


def assemble(records, num_obs, threshold_obs, variant="static"):
    """rank-0 side of the sweep point: sort the gathered records by episode, apply the acceptance filter of S/main_mpc.py:121-128
    (D/main_mpc.py:137-148) in episode order and build the arrays the reference saves"""
    rec = records[np.argsort(records[:, 0], kind="stable")]
    init_state, _, _, _ = scenes.driver_inputs(variant)
    keep = [r for r in rec if r[1] <= threshold_obs]
    cx = np.zeros((0, 11)); cy = np.zeros((0, 11)); ist = np.zeros((0, 6))
    xo = np.zeros((0, num_obs)); yo = np.zeros((0, num_obs)); vxo = np.zeros((0, num_obs)); vyo = np.zeros((0, num_obs))
    pso = np.zeros((0, num_obs)); xt_all = np.zeros((0, num_obs, 100)); yt_all = np.zeros((0, num_obs, 100))
    for r in keep:
        if variant == "dynamic":
            (x, y, vx, vy, psi), _, xt, yt = scenes.dynamic_scene(num_obs, int(r[0]))
            pso = np.append(pso, psi.reshape(1, -1), axis=0)
            xt_all = np.append(xt_all, xt.reshape(1, num_obs, -1), axis=0); yt_all = np.append(yt_all, yt.reshape(1, num_obs, -1), axis=0)
        else:
            (x, y, vx, vy, _), _ = scenes.static_scene(num_obs, int(r[0]))
        cx = np.append(cx, r[3:14].reshape(1, -1), axis=0); cy = np.append(cy, r[14:25].reshape(1, -1), axis=0)
        ist = np.append(ist, np.asarray(init_state).reshape(1, -1), axis=0)
        xo = np.append(xo, x.reshape(1, -1), axis=0); yo = np.append(yo, y.reshape(1, -1), axis=0)
        vxo = np.append(vxo, vx.reshape(1, -1), axis=0); vyo = np.append(vyo, vy.reshape(1, -1), axis=0)
    out = dict(cx=cx, cy=cy, init_state=ist, x_obs=xo, y_obs=yo, vx_obs=vxo, vy_obs=vyo)
    if variant == "dynamic":
        out.update(psi_obs=pso, x_obs_traj=xt_all, y_obs_traj=yt_all)
    return out


def kernel_tag(kernel, cost):
    """extra arrays of a data file: an MMD plan made with a non-reference kernel says so"""
    return dict(kernel=kernel) if kernel != "laplace" and cost in ("mmd_opt", "mmd_random") else {}


def data_path(root, noise, noise_level, num_prime, cost, num_reduced, num_obs):
    return os.path.join(root, "{}_noise".format(noise), "noise_{}".format(int(noise_level * 100)), "ts_{}".format(num_prime),
                        "{}_{}_samples_{}_obs".format(cost, num_reduced, num_obs))


def run_sweep(args, rank=0, world=1, gather=None, device=0, log=print):
    """`gather(records) -> all records on rank 0` is the only cross-rank exchange (torch.distributed all_gather in __main__)."""
    written = []
    kernel = getattr(args, "kernel", "laplace")
    for noise in args.noises:
        for noise_level in args.noise_levels:
            for num_prime in args.num_prime:
                for num_obs in args.num_obs:
                    for num_reduced in args.num_reduced_sets:
                        mine = shard(args.num_configs, rank, world)
                        prob = CEM(num_reduced, num_obs, noise_level, num_prime, noise, args.acc_const_noise, args.steer_const_noise,
                                   variant=args.variant, max_episodes=max(len(mine), 1), device=device, kernel=kernel)
                        batch = scenes.static_batch(prob, mine, args.variant)
                        for cost in args.costs:
                            _, threshold_obs = thresholds(prob, cost)
                            t0 = time.time()
                            out = prob.solve_batch(solve_cost(cost), **batch) if mine else None
                            rec = pack_records(mine, out) if mine else np.zeros((0, 26), F32)
                            if gather is not None:
                                rec = gather(rec)
                            if rank == 0:
                                arrays = assemble(rec, num_obs, threshold_obs, args.variant)
                                arrays.update(kernel_tag(kernel, cost))
                                path = data_path(args.root, noise, noise_level, num_prime, cost, num_reduced, num_obs)
                                os.makedirs(os.path.dirname(path), exist_ok=True)
                                np.savez(path, **arrays)
                                written.append(path + ".npz")
                                log("cost {}, reduced_set {}, num_obs {}, num_prime {}, noise_level {}, noise {}: {} of {} accepted, {:.2f} s".format(
                                    cost, num_reduced, num_obs, num_prime, noise_level, noise, arrays["cx"].shape[0], args.num_configs, time.time() - t0))
                        del prob
    return written


def dist_gather(rec, world, device):
    """all ranks' records, concatenated in rank order (ragged: shards differ by at most one episode).  The one collective of the sweep."""
    import torch
    import torch.distributed as dist
    n = torch.tensor([rec.shape[0]], device=device); ns = [torch.zeros_like(n) for _ in range(world)]
    dist.all_gather(ns, n)
    m = int(max(int(v.item()) for v in ns))
    pad = torch.zeros((m, 26), device=device); pad[:rec.shape[0]] = torch.as_tensor(rec, device=device)
    bufs = [torch.zeros_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad)
    return np.concatenate([b[:int(k.item())].cpu().numpy() for b, k in zip(bufs, ns)], 0)


def build_parser():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--noise_levels", type=float, nargs="+", required=True)
    p.add_argument("--num_reduced_sets", type=int, nargs="+", required=True)
    p.add_argument("--num_obs", type=int, nargs="+", required=True)
    p.add_argument("--costs", type=str, nargs="+", required=True)
    p.add_argument("--num_prime", type=int, nargs="+", required=True)
    p.add_argument("--noises", type=str, nargs="+", required=True)
    p.add_argument("--acc_const_noise", type=float, required=True)
    p.add_argument("--steer_const_noise", type=float, required=True)
    p.add_argument("--num_configs", type=int, default=200, help="episodes per sweep point (main_mpc.py:76)")
    p.add_argument("--root", type=str, default="./data")
    p.add_argument("--variant", type=str, default="static", choices=["static", "dynamic"])
    p.add_argument("--kernel", type=str, default="laplace", choices=["laplace", "gaussian"],
                   help="kernel of the mmd_opt / mmd_random risk cost (default: laplace, the reference's)")
    return p


def main(argv=None, variant=None):
    args = build_parser().parse_args(argv)
    if variant is not None:
        args.variant = variant
    rank, world, local = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("LOCAL_RANK", "0"))
    gather = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        gather = lambda rec: dist_gather(rec, world, "cuda")
    run_sweep(args, rank, world, gather, device=local)
    if world > 1:
        import torch.distributed as dist
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
