"""Monte-Carlo validation of the planned trajectories: the reference's `validation.py` workflow (synthetic_static_obs/validation.py,
synthetic_dynamic_obs/validation.py) with the 1000-rollout evaluation of `compute_stats` on the GPU.

What stays on the host, and why: the reference seeds NumPy's legacy global stream per trajectory (`np.random.seed(key)`, validation.py:43)
and draws `multivariate_normal` / `beta` from it (:65-84).  Bit-identical collision counts need those exact MT19937 draws, so the noise is
drawn here with the same calls in the same order, the controls are perturbed in float64 exactly as the reference does, and the perturbed
controls go to `mpcmmd_validate_host` (csrc/k_validate.cuh), which rolls the 1000 bicycle models out and counts intersections.
Opt-in (`--rng device`, `compute_stats_batch(..., rng="device")`): the same legacy stream restated on the GPU (csrc/dnprng.cuh,
k_validate_noise.cuh), one stream per trajectory.  Its stream consumption is NumPy's exactly; its values differ from NumPy's only where
CUDA's double pow / log / exp round differently from glibc's (DESIGN.md section 3 item 6).  The host draws stay the default and the reference.
Opt-in (`--rng jax`, `compute_stats_batch(..., rng="jax")`): counter-based noise from the JAX protocol the reference's solver draws with
(csrc/drng.cuh, k_validate_jax.cuh, DESIGN.md section 3 item 7), drawn by each rollout on the GPU as it rolls out.  Same distributions,
different random numbers: its counts estimate what the reference's estimate, for any number of rollouts (`--num_rollouts`).

Same command line as the reference, same input files (`./data/{noise}_noise/noise_{L}/ts_{np}/{cost}_{nr}_samples_{O}_obs.npz`), same output
(`./stats/{noise}_noise/noise_{L}/ts_{np}/{nr}_samples_{O}_obs.npz` with coll_cvar, coll_cvar_lane, coll_mmd_opt, coll_mmd_opt_lane,
coll_mmd_random, coll_mmd_random_lane; with `--rng jax` or a non-default `--num_rollouts` also rng and num_rollouts, so those counts are
not taken for the reference's; when the mmd_opt plans carry `kernel` (driver `--kernel gaussian`), so does the stats file; with `--risk`
also each plan's Monte-Carlo risk, `risk_stats_batch`).  Trajectory pairs are enumerated exactly like the reference does -- `set(cvar rows) & set(mmd_opt rows)`
in Python set-iteration order, position k in that order is the RNG seed of the pair (SURVEY.md Q21) -- so the per-pair draws are the same.
"""
from __future__ import annotations

import argparse
import ctypes as C
import os

import numpy as np

from . import binding as B
from .cem_impl import CEM

NUM_ROLLOUTS = 1000          # _num_batch, validation.py:173


def compute_controls(prob, cx, cy):
    """acc (101,), steer (100,) of the planned trajectory in float64 (validation.py:126-132,141-148): np.dot of the float32 basis with the
    float64 coefficients promotes to float64."""
    cx, cy = np.asarray(cx, np.float64).reshape(-1), np.asarray(cy, np.float64).reshape(-1)
    Pdot, Pddot = np.asarray(prob.Pdot_jax), np.asarray(prob.Pddot_jax)
    xdot, xddot = np.dot(Pdot, cx), np.dot(Pddot, cx)
    ydot, yddot = np.dot(Pdot, cy), np.dot(Pddot, cy)
    v = np.sqrt(xdot ** 2 + ydot ** 2)
    v = np.hstack((v, v[-1]))
    acc = np.diff(v) / prob.t
    acc = np.hstack((acc, acc[-1]))
    curvature = (yddot * xdot - ydot * xddot) / ((xdot ** 2 + ydot ** 2) ** (1.5))
    steer = np.arctan(curvature * prob.wheel_base)
    return acc, steer


def perturbed_controls(prob, acc, steer, noise_level, num_prime, noise, key, n_roll=NUM_ROLLOUTS):
    """the noisy control sequences of `compute_rollout_complete` (validation.py:40-90): legacy-stream draws in the reference's order,
    float64.  acc, steer: the first num_prime planned controls.  Returns (n_roll, num_prime) x2."""
    np.random.seed(key)
    if noise == "gaussian":
        z_acc = np.random.multivariate_normal(np.zeros(num_prime), np.eye(num_prime), (n_roll,))
        z_steer = np.random.multivariate_normal(np.zeros(num_prime), np.eye(num_prime), (n_roll,))
        acc_pert = noise_level * np.abs(acc) * z_acc
        steer_pert = noise_level * np.abs(steer) * z_steer
    else:
        b_acc = np.random.beta(prob.beta_a * np.abs(acc), prob.beta_b * np.abs(acc), (n_roll, num_prime))
        b_steer = np.random.beta(prob.beta_a * np.abs(steer) + 1e-5, prob.beta_b * np.abs(steer) + 1e-5, (n_roll, num_prime))
        acc_pert = noise_level * (2 * b_acc - 1)
        steer_pert = prob.cem_helper.K_steer * noise_level * (2 * b_steer - 1)
    z = np.random.multivariate_normal(np.zeros(num_prime), np.eye(num_prime), (n_roll,))
    return acc + acc_pert + prob.acc_const_noise * z, steer + steer_pert + prob.steer_const_noise * z


def _host_draws(prob, items, acc_p, steer_p, noise_level, num_prime, noise, n_roll):
    """perturbed_controls of every item from its planned controls acc_p[i], steer_p[i] and seed item["key"]: (n, n_roll, num_prime) x2"""
    acc = np.empty((len(items), n_roll, num_prime)); steer = np.empty((len(items), n_roll, num_prime))
    for i, it in enumerate(items):
        acc[i], steer[i] = perturbed_controls(prob, acc_p[i], steer_p[i], noise_level, num_prime, noise, it["key"], n_roll)
    return acc, steer


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _device_index(prob, device):
    """the CUDA device of a call: `device` if given, else the handle's"""
    return (prob.device.index if device is None else int(device)) or 0


def _geometry(prob):
    """dt, wheel_base, a_obs, b_obs, y_lb, y_ub: the rollout and cost arguments of every validation entry point"""
    return float(prob.t), float(prob.wheel_base), float(prob.a_obs), float(prob.b_obs), float(prob.y_lb), float(prob.y_ub)


def _noise_args(prob, noise, noise_level):
    """noise_kind, noise_level, K_steer, beta_a, beta_b, acc_const_noise, steer_const_noise: the noise arguments of the entry points that
    draw on the device"""
    return (B.NOISE_KINDS[noise], float(noise_level), float(prob.cem_helper.K_steer), float(prob.beta_a), float(prob.beta_b),
            float(prob.acc_const_noise), float(prob.steer_const_noise))


def _check_noise(noise):
    if noise not in B.NOISE_KINDS:
        raise ValueError("noise must be one of %s, not %r" % (sorted(B.NOISE_KINDS), noise))


def _check_n_roll(n_roll, num_prime, why=""):
    """n_roll an integer >= 1 with n_roll * num_prime below 2**31; `why` closes the second message"""
    if isinstance(n_roll, bool) or not isinstance(n_roll, (int, np.integer)) or n_roll < 1:
        raise ValueError("n_roll must be an integer >= 1, not %r" % (n_roll,))
    if int(n_roll) * int(num_prime) >= 2 ** 31:
        raise ValueError("n_roll * num_prime must be below 2**31" + why)


def _inputs(prob, items, num_prime, num_obs):
    """per-trajectory inputs of the validation entry points: planned controls (n, num_prime) x2, state0 (n, 5), obstacle trajectories
    (n, num_obs, num_prime) x2, and whether the obstacle cost is float32 (static variant)"""
    n = len(items)
    acc_p = np.empty((n, num_prime)); steer_p = np.empty((n, num_prime))
    state0 = np.empty((n, 5)); xo = np.empty((n, num_obs, num_prime)); yo = np.empty((n, num_obs, num_prime))
    static = "x_obs_traj" not in items[0]
    for i, it in enumerate(items):
        acc, steer = compute_controls(prob, it["cx"], it["cy"])
        acc_p[i], steer_p[i] = acc[0:num_prime], steer[0:num_prime]
        s = np.asarray(it["init_state"], np.float64).reshape(-1)
        state0[i] = [s[0], s[1], s[2], s[3], np.arctan2(s[3], s[2])]
        if static:
            x_obs, y_obs = np.asarray(it["x_obs"]).reshape(-1), np.asarray(it["y_obs"]).reshape(-1)
            vx_obs, vy_obs = np.asarray(it["vx_obs"]).reshape(-1), np.asarray(it["vy_obs"]).reshape(-1)
            xt, yt, _ = prob.cem_helper.compute_obs_trajectories(x_obs, y_obs, vx_obs, vy_obs, np.arctan2(vy_obs, vx_obs))   # float32
        else:
            xt = np.asarray(it["x_obs_traj"]).reshape(num_obs, prob.num); yt = np.asarray(it["y_obs_traj"]).reshape(num_obs, prob.num)
        xo[i] = xt[:, 0:num_prime]; yo[i] = yt[:, 0:num_prime]
    return acc_p, steer_p, state0, xo, yo, static


def compute_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, want_rollouts=False, device=None, n_roll=NUM_ROLLOUTS, rng="host"):
    """`compute_stats` (validation.py:134-171) for a list of trajectories in ONE device call.

    items: dicts with cx, cy (11,), init_state (6,), key, and either x_obs, y_obs, vx_obs, vy_obs (static variant) or
    x_obs_traj, y_obs_traj (num_obs, 100) (dynamic variant).  Returns count (n,), count_lane (n,) int arrays [, x_roll, y_roll].

    rng="host" (default) draws the noise from NumPy's legacy stream here, exactly as the reference does.  rng="device" draws the same
    stream on the GPU (`seeded_stats_batch`): identical stream consumption, values within CUDA's libm rounding of NumPy's.  rng="jax"
    draws counter-based JAX-protocol noise in the rollout kernel (`threefry_stats_batch`): not NumPy's numbers, same distributions.
    Neither returns rollouts."""
    if rng in ("device", "jax"):
        if want_rollouts:
            raise ValueError("compute_stats_batch: want_rollouts needs rng='host'")
        f = seeded_stats_batch if rng == "device" else threefry_stats_batch
        return f(prob, items, num_prime, noise_level, noise, num_obs, device=device, n_roll=n_roll)[:2]
    if rng != "host":
        raise ValueError("compute_stats_batch: rng must be 'host', 'device' or 'jax', not %r" % (rng,))
    n = len(items)
    if n == 0:
        z = np.zeros(0, np.int64)
        return (z, z, None, None) if want_rollouts else (z, z)
    acc_p, steer_p, state0, xo, yo, static = _inputs(prob, items, num_prime, num_obs)
    acc_all, steer_all = _host_draws(prob, items, acc_p, steer_p, noise_level, num_prime, noise, n_roll)
    count = np.zeros(n, np.int32); lane = np.zeros(n, np.int32)
    xr = np.empty((n, n_roll, num_prime)) if want_rollouts else None
    yr = np.empty((n, n_roll, num_prime)) if want_rollouts else None
    B.check(B.load().mpcmmd_validate_host(_device_index(prob, device), n, n_roll, num_prime, num_obs, 1 if static else 0, *_geometry(prob),
                                          _ptr(acc_all), _ptr(steer_all), _ptr(state0), _ptr(xo), _ptr(yo), _ptr(count), _ptr(lane), _ptr(xr),
                                          _ptr(yr)))
    return (count, lane, xr, yr) if want_rollouts else (count, lane)


STATE_WORDS = 628                 # key[624], pos, has_gauss, cached gauss as float64 bits (mpcmmd_validate_seeded_host's state_out)
_IDENTITY_OK = {}


def _mvn_identity_is_exact(num_prime):
    """multivariate_normal(0, I) multiplies the standard normals by sqrt(s)[:, None] * vh of svd(I) (NumPy's legacy
    multivariate_normal); the device path draws plain standard normals, which is the same stream only if that factor is exactly I.
    Checked once per num_prime against the LAPACK NumPy runs on."""
    if num_prime not in _IDENTITY_OK:
        _, s, vh = np.linalg.svd(np.eye(num_prime))
        _IDENTITY_OK[num_prime] = bool(np.array_equal(np.sqrt(s)[:, None] * vh, np.eye(num_prime)))
    return _IDENTITY_OK[num_prime]


def check_beta_params(prob, acc, steer):
    """the argument check np.random.beta makes before it draws (NaN passes): ValueError("a <= 0") / ("b <= 0") for the first failing
    call of perturbed_controls -- the acceleration draw, then the steering draw"""
    for a, b in ((prob.beta_a * np.abs(acc), prob.beta_b * np.abs(acc)), (prob.beta_a * np.abs(steer) + 1e-5, prob.beta_b * np.abs(steer) + 1e-5)):
        if np.any(np.less_equal(a, 0)):
            raise ValueError("a <= 0")
        if np.any(np.less_equal(b, 0)):
            raise ValueError("b <= 0")


def _seeds(items):
    """the per-trajectory seeds as uint32, refused outside np.random.seed's range"""
    seeds = np.empty(len(items), np.uint32)
    for i, it in enumerate(items):
        k = int(it["key"])
        if not 0 <= k <= 0xffffffff:
            raise ValueError("Seed must be between 0 and 2**32 - 1")                  # np.random.seed's range
        seeds[i] = k
    return seeds


def seeded_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, want_draws=False, device=None, n_roll=NUM_ROLLOUTS):
    """`compute_stats_batch` with the legacy-stream noise drawn on the GPU (mpcmmd_validate_seeded_host, csrc/k_validate_noise.cuh):
    the planned controls are computed here, each trajectory's stream is np.random.seed(item["key"]) restated on the device.
    Returns count, count_lane (n,) [, acc, steer (n, n_roll, num_prime) perturbed controls, state (n, 628) uint32 streams after the
    last draw = np.random.get_state()[1:] packed as key[624], pos, has_gauss, gauss bits]."""
    _check_noise(noise)
    n = len(items)
    if n == 0:
        z = np.zeros(0, np.int64)
        return (z, z, np.zeros((0, n_roll, num_prime)), np.zeros((0, n_roll, num_prime)), np.zeros((0, STATE_WORDS), np.uint32)) if want_draws else (z, z)
    seeds = _seeds(items)
    if not _mvn_identity_is_exact(num_prime):
        raise RuntimeError("multivariate_normal(0, eye(%d)) is not exactly standard_normal with this LAPACK: use rng='host'" % num_prime)
    acc_p, steer_p, state0, xo, yo, static = _inputs(prob, items, num_prime, num_obs)
    if noise == "beta":
        for i in range(n):
            check_beta_params(prob, acc_p[i], steer_p[i])
    count = np.zeros(n, np.int32); lane = np.zeros(n, np.int32)
    acc = np.empty((n, n_roll, num_prime)) if want_draws else None
    steer = np.empty((n, n_roll, num_prime)) if want_draws else None
    state = np.empty((n, STATE_WORDS), np.uint32) if want_draws else None
    B.check(B.load().mpcmmd_validate_seeded_host(
        _device_index(prob, device), n, n_roll, num_prime, num_obs, 1 if static else 0, *_noise_args(prob, noise, noise_level), *_geometry(prob),
        _ptr(seeds), _ptr(acc_p), _ptr(steer_p), _ptr(state0), _ptr(xo), _ptr(yo), _ptr(count), _ptr(lane), _ptr(acc), _ptr(steer), _ptr(state)))
    return (count, lane, acc, steer, state) if want_draws else (count, lane)


def threefry_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, want_draws=False, device=None, n_roll=NUM_ROLLOUTS):
    """`compute_stats_batch` with counter-based noise (mpcmmd_validate_threefry_host, csrc/k_validate_jax.cuh; DESIGN.md section 3
    item 7): trajectory i's noise is JAX's random.beta / random.normal of split(PRNGKey(item["key"]), 3) over an (n_roll, num_prime)
    array, drawn by each rollout as it rolls out.  No shape parameter check (JAX makes none: at num_prime = 100 the acceleration
    draws of the last knot are NaN and reach only the discarded final state).  Returns count, count_lane (n,) [, acc, steer
    (n, n_roll, num_prime) perturbed controls]."""
    _check_noise(noise)
    _check_n_roll(n_roll, num_prime, " (JAX's uint32 element counters)")
    n = len(items)
    if n == 0:
        z = np.zeros(0, np.int64)
        return (z, z, np.zeros((0, n_roll, num_prime)), np.zeros((0, n_roll, num_prime))) if want_draws else (z, z)
    seeds = _seeds(items)
    acc_p, steer_p, state0, xo, yo, static = _inputs(prob, items, num_prime, num_obs)
    count = np.zeros(n, np.int32); lane = np.zeros(n, np.int32)
    acc = np.empty((n, n_roll, num_prime)) if want_draws else None
    steer = np.empty((n, n_roll, num_prime)) if want_draws else None
    B.check(B.load().mpcmmd_validate_threefry_host(
        _device_index(prob, device), n, int(n_roll), num_prime, num_obs, 1 if static else 0, *_noise_args(prob, noise, noise_level), *_geometry(prob),
        _ptr(seeds), _ptr(acc_p), _ptr(steer_p), _ptr(state0), _ptr(xo), _ptr(yo), _ptr(count), _ptr(lane), _ptr(acc), _ptr(steer)))
    return (count, lane, acc, steer) if want_draws else (count, lane)


RISK_KEYS = ("p_coll", "p_lane", "mean_obs", "var_obs", "cvar_obs")


def _check_alpha(alpha):
    a = float(alpha)
    if not 0.0 <= a <= 1.0:
        raise ValueError("alpha must lie in [0, 1], not %r" % (alpha,))
    return a


def _check_sigma(sigma, n):
    """sigma as a float64 (n,) array: one Laplace bandwidth per plan (a scalar applies to every plan), each > 0 and finite"""
    sg = np.asarray(sigma, np.float64)
    if sg.ndim == 0:
        sg = np.full(n, float(sg))
    if sg.shape != (n,):
        raise ValueError("sigma must be a scalar or have shape (%d,), not %s" % (n, sg.shape))
    if not np.all(np.isfinite(sg) & (sg > 0)):
        raise ValueError("sigma must be positive and finite")
    return np.ascontiguousarray(sg)


def _risk_struct(shape, alpha, ker_wt, sigma, costs_shape=None):
    """(mpcmmd_risk_out, its output arrays): statistics of `shape`, per-rollout costs of costs_shape if given"""
    out = {k: np.zeros(shape) for k in RISK_KEYS}
    if sigma is not None:
        out["mmd_obs"] = np.zeros(shape)
    if costs_shape is not None:
        out["c_obs"], out["c_lane"] = np.zeros(costs_shape), np.zeros(costs_shape)
    p = lambda k: out[k].ctypes.data if k in out else None
    r = B.MpcmmdRiskOut(alpha, float(ker_wt), None if sigma is None else sigma.ctypes.data, *[p(k) for k in RISK_KEYS + ("mmd_obs", "c_obs", "c_lane")])
    return r, out


def risk_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, n_roll=NUM_ROLLOUTS, rng="host", alpha=0.98, sigma=None,
                     want_rollout_costs=False, device=None):
    """Monte-Carlo risk of each plan (DESIGN.md section 3 item 9): the rollouts of `compute_stats_batch` with rng="host" (NumPy's legacy
    stream, mpcmmd_validate_risk_host) or rng="jax" (counter-based noise, mpcmmd_validate_threefry_risk_host), and per plan the collision
    and lane probabilities (a NaN cost counts as a hit), the mean, VaR_alpha and CVaR_alpha of the obstacle cost, and with `sigma` (one
    Laplace bandwidth per plan, or a scalar) its MMD ker_wt (E k(c, c') - 2 E k(c, 0)), ker_wt = prob.ker_wt.
    Returns a dict: count, count_lane (as compute_stats_batch), p_coll, p_lane, mean_obs, var_obs, cvar_obs (n,) [, mmd_obs (n,)]
    [, c_obs, c_lane (n, n_roll) per-rollout costs]."""
    if rng == "device":
        raise ValueError("risk_stats_batch: rng='device' has no risk statistics (its draws are NumPy's: use rng='host')")
    if rng not in ("host", "jax"):
        raise ValueError("risk_stats_batch: rng must be 'host' or 'jax', not %r" % (rng,))
    _check_noise(noise)
    _check_n_roll(n_roll, num_prime)
    alpha = _check_alpha(alpha)
    n = len(items)
    if sigma is not None:
        if getattr(prob, "kernel", "laplace") != "laplace":
            raise ValueError("risk_stats_batch: the Monte-Carlo MMD is the Laplace kernel's; this handle uses kernel=%r" % (prob.kernel,))
        sigma = _check_sigma(sigma, n)
    seeds = _seeds(items)
    n_roll = int(n_roll)
    r, out = _risk_struct(n, alpha, getattr(prob, "ker_wt", 1000.0), sigma, (n, n_roll) if want_rollout_costs else None)
    count = np.zeros(n, np.int32); lane = np.zeros(n, np.int32)
    out.update(count=count, count_lane=lane)
    if n == 0:
        return out
    acc_p, steer_p, state0, xo, yo, static = _inputs(prob, items, num_prime, num_obs)
    dev = _device_index(prob, device)
    if rng == "host":
        acc_all, steer_all = _host_draws(prob, items, acc_p, steer_p, noise_level, num_prime, noise, n_roll)
        B.check(B.load().mpcmmd_validate_risk_host(dev, n, n_roll, num_prime, num_obs, 1 if static else 0, *_geometry(prob), _ptr(acc_all),
                                                   _ptr(steer_all), _ptr(state0), _ptr(xo), _ptr(yo), _ptr(count), _ptr(lane), C.byref(r)))
    else:
        B.check(B.load().mpcmmd_validate_threefry_risk_host(
            dev, n, n_roll, num_prime, num_obs, 1 if static else 0, *_noise_args(prob, noise, noise_level), *_geometry(prob), _ptr(seeds),
            _ptr(acc_p), _ptr(steer_p), _ptr(state0), _ptr(xo), _ptr(yo), _ptr(count), _ptr(lane), C.byref(r)))
    return out


def risk_stats(c_obs, c_lane=None, alpha=0.98, sigma=None, ker_wt=1000.0, device=0):
    """the risk statistics of given per-rollout costs (mpcmmd_risk_stats_host): c_obs (n,) or (n_sets, n), each >= 0 and finite or NaN;
    c_lane the same shape or None (p_lane = 0); sigma a scalar or one bandwidth per set.  Returns a dict of arrays of shape c_obs.shape[:-1]:
    p_coll, p_lane, mean_obs, var_obs, cvar_obs [, mmd_obs]."""
    co = np.ascontiguousarray(c_obs, np.float64)
    if co.ndim not in (1, 2) or co.shape[-1] < 1 or co.size == 0:
        raise ValueError("c_obs must have shape (n,) or (n_sets, n) with n >= 1, not %s" % (co.shape,))
    if np.any(co < 0) or np.any(np.isinf(co)):
        raise ValueError("c_obs values must be >= 0 and finite, or NaN")
    cl = None
    if c_lane is not None:
        cl = np.ascontiguousarray(c_lane, np.float64)
        if cl.shape != co.shape:
            raise ValueError("c_lane must have the shape of c_obs %s, not %s" % (co.shape, cl.shape))
    shape = co.shape[:-1]
    n_sets, n = (1, co.shape[0]) if co.ndim == 1 else co.shape
    alpha = _check_alpha(alpha)
    if sigma is not None:
        sigma = _check_sigma(np.reshape(sigma, -1) if np.ndim(sigma) else sigma, n_sets)
    r, out = _risk_struct(shape, alpha, ker_wt, sigma)
    B.check(B.load().mpcmmd_risk_stats_host(int(device), n_sets, n, _ptr(co), _ptr(cl), C.byref(r)))
    return out


def _load(root, noise, noise_level, num_prime, cost, num_reduced, num_obs):
    return np.load(root + "/{}_noise/noise_{}/ts_{}/{}_{}_samples_{}_obs.npz".format(noise, int(noise_level * 100), num_prime, cost, num_reduced, num_obs))


def _matrix(d, num_obs):
    return np.hstack((np.asarray(d["init_state"]), np.asarray(d["x_obs"])[:, 0:num_obs], np.asarray(d["y_obs"])[:, 0:num_obs],
                      np.asarray(d["vx_obs"])[:, 0:num_obs], np.asarray(d["vy_obs"])[:, 0:num_obs]))


def matched_pairs(data_cvar, data_mmd_opt, num_obs):
    """[(k, idx_cvar, idx_mmd_opt)]: scenes solved by BOTH costs, in the reference's order (validation.py:290-313): Python set iteration
    order of `cset & dset`; the first matching row of each file."""
    cvar_matrix, mmd_opt_matrix = _matrix(data_cvar, num_obs), _matrix(data_mmd_opt, num_obs)
    cset = set([tuple(x) for x in cvar_matrix])
    dset = set([tuple(x) for x in mmd_opt_matrix])
    eset = np.array([x for x in cset & dset])
    out = []
    for k in range(0, eset.shape[0]):
        idx_cvar = np.where(np.all(eset[k] == cvar_matrix, axis=1))[0]
        idx_mmd_opt = np.where(np.all(eset[k] == mmd_opt_matrix, axis=1))[0]
        out.append((k, int(idx_cvar[0]), int(idx_mmd_opt[0])))
    return out


def _item(d, idx, key, dynamic):
    it = dict(cx=np.asarray(d["cx"])[idx], cy=np.asarray(d["cy"])[idx], init_state=np.asarray(d["init_state"])[idx], key=key)
    if dynamic:
        it.update(x_obs_traj=np.asarray(d["x_obs_traj"])[idx], y_obs_traj=np.asarray(d["y_obs_traj"])[idx])
    else:
        it.update(x_obs=np.asarray(d["x_obs"])[idx], y_obs=np.asarray(d["y_obs"])[idx], vx_obs=np.asarray(d["vx_obs"])[idx], vy_obs=np.asarray(d["vy_obs"])[idx])
    return it


def run_validation(args, variant="static", device=0, log=print):
    risk = getattr(args, "risk", False)
    if risk and args.rng not in ("host", "jax"):
        raise ValueError("--risk needs --rng host or --rng jax (the legacy-stream device draws are NumPy's: use --rng host)")
    written = []
    dynamic = variant == "dynamic"
    for noise in args.noises:
        for noise_level in args.noise_levels:
            for num_prime in args.num_prime:
                for num_obs in args.num_obs:
                    for num_reduced in args.num_reduced_sets:
                        prob = CEM(num_reduced, num_obs, noise_level, num_prime, noise, args.acc_const_noise, args.steer_const_noise,
                                   variant=variant, max_episodes=1, device=device)
                        data_mmd_opt = _load(args.root, noise, noise_level, num_prime, "mmd_opt", num_reduced, num_obs)
                        data_cvar = _load(args.root, noise, noise_level, num_prime, "cvar", num_reduced, num_obs)
                        pairs = matched_pairs(data_cvar, data_mmd_opt, num_obs)
                        log((len(pairs), _matrix(data_cvar, num_obs).shape[1]))                     # the reference prints eset.shape
                        # both costs of a scene share the seed k (validation.py:315-336)
                        items = [_item(data_mmd_opt, im, k, dynamic) for k, _, im in pairs] + [_item(data_cvar, ic, k, dynamic) for k, ic, _ in pairs]
                        extra = {}
                        if risk:
                            rs = risk_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, n_roll=args.num_rollouts, rng=args.rng,
                                                  alpha=args.risk_alpha)
                            count, lane = rs["count"], rs["count_lane"]
                        else:
                            count, lane = compute_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, n_roll=args.num_rollouts, rng=args.rng)
                        m = len(pairs)
                        if risk:                                  # the same order as the coll_* arrays: pair k at position k
                            extra["risk_alpha"] = float(args.risk_alpha)
                            for k in RISK_KEYS:
                                extra[k + "_cvar"], extra[k + "_mmd_opt"] = rs[k][m:], rs[k][:m]
                        f = lambda a: np.asarray(a, np.float64)                                   # np.append([], int) yields float64 arrays
                        path = "{}/{}_noise/noise_{}/ts_{}/{}_samples_{}_obs".format(args.stats_root, noise, int(noise_level * 100), num_prime, num_reduced, num_obs)
                        os.makedirs(os.path.dirname(path), exist_ok=True)
                        # counts that are not the reference's estimator (other noise or other rollout count) say so in the file
                        tag = dict(rng=args.rng, num_rollouts=args.num_rollouts) if args.rng == "jax" or args.num_rollouts != NUM_ROLLOUTS else {}
                        if "kernel" in data_mmd_opt.files:                                        # plans made with a non-reference MMD kernel
                            tag["kernel"] = str(data_mmd_opt["kernel"])
                        np.savez(path, coll_cvar=f(count[m:]), coll_cvar_lane=f(lane[m:]), coll_mmd_opt=f(count[:m]), coll_mmd_opt_lane=f(lane[:m]),
                                 coll_mmd_random=[], coll_mmd_random_lane=[], **tag, **extra)
                        written.append(path + ".npz")
                        del prob
    return written


def build_parser():
    p = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    p.add_argument("--noise_levels", type=float, nargs="+", required=True)
    p.add_argument("--num_reduced_sets", type=int, nargs="+", required=True)
    p.add_argument("--num_obs", type=int, nargs="+", required=True)
    p.add_argument("--num_prime", type=int, nargs="+", required=True)
    p.add_argument("--noises", type=str, nargs="+", required=True)
    p.add_argument("--acc_const_noise", type=float, required=True)
    p.add_argument("--steer_const_noise", type=float, required=True)
    p.add_argument("--root", type=str, default="./data")
    p.add_argument("--stats_root", type=str, default="./stats")
    p.add_argument("--variant", type=str, default="static", choices=["static", "dynamic"])
    p.add_argument("--rng", type=str, default="host", choices=["host", "device", "jax"],
                   help="host (default): NumPy's legacy stream, as the reference; device: the same stream drawn on the GPU (identical "
                        "consumption, values within CUDA's pow / log / exp rounding); jax: counter-based JAX-protocol noise drawn by each "
                        "rollout on the GPU (same distributions, not the reference's numbers)")
    p.add_argument("--num_rollouts", type=_positive_int, default=NUM_ROLLOUTS,
                   help="noisy rollouts per planned trajectory (default %d, the reference's _num_batch)" % NUM_ROLLOUTS)
    p.add_argument("--risk", action="store_true",
                   help="also write each plan's Monte-Carlo risk: p_coll_*, p_lane_*, mean_obs_*, var_obs_*, cvar_obs_* and risk_alpha "
                        "(needs --rng host or jax)")
    p.add_argument("--risk_alpha", type=_unit_float, default=0.98, help="VaR / CVaR level of --risk (default 0.98, the solver's alpha_quant)")
    return p


def _unit_float(s):
    v = float(s)
    if not 0.0 <= v <= 1.0:
        raise argparse.ArgumentTypeError("must lie in [0, 1], not %s" % s)
    return v


def _positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be >= 1, not %d" % v)
    return v


def main(argv=None, variant=None):
    parser = build_parser()
    args = parser.parse_args(argv)
    if args.risk and args.rng == "device":
        parser.error("--risk needs --rng host or --rng jax")
    run_validation(args, variant or args.variant)


if __name__ == "__main__":
    main()
