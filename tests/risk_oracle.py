"""CPU restatement of the Monte-Carlo risk statistics (DESIGN.md section 3 item 9) -- TEST INFRASTRUCTURE ONLY, never imported by the
product path.  It states the definitions literally, next to oracle/oracle_validation.py's `counts` (whose dtype rule it shares):

    rollout_costs   per-rollout obstacle cost c_obs = max over (obstacle, t) of max(0, cost), lane cost c_lane = max_t lb + max_t ub
    risk_stats      p_coll, p_lane, mean, VaR (cvar_cost's quantile expression in float64 on np.sort), CVaR, MMD (O(n^2) double sum)
    mmd_sum_recurrence   the all-pairs Laplace sum S from the sorted costs in O(n): P_{i+1} = (P_i + 1) exp(-(v_{i+1} - v_i) / sigma)
"""
import math

import numpy as np

f32 = np.float32


def rollout_costs(x_roll, y_roll, x_obs_traj, y_obs_traj, num_prime, a_obs, b_obs, y_lb, y_ub, obs_f32):
    """c_obs, c_lane (n_roll,) float64 of one plan's rollouts x_roll, y_roll (n_roll, num_prime): the cost expressions of `counts`"""
    xo, yo = np.asarray(x_obs_traj)[:, 0:num_prime][:, None], np.asarray(y_obs_traj)[:, 0:num_prime][:, None]
    if obs_f32:
        wc, ws = x_roll.astype(f32) - xo.astype(f32), y_roll.astype(f32) - yo.astype(f32)
        cost = -(wc * wc) / f32(a_obs ** 2) - (ws * ws) / f32(b_obs ** 2) + f32(1.0)
    else:
        wc, ws = x_roll - xo, y_roll - yo
        cost = -(wc ** 2) / (a_obs ** 2) - (ws ** 2) / (b_obs ** 2) + 1.0
    c_obs = np.max(np.maximum(np.zeros_like(cost), cost), axis=(0, 2)).astype(np.float64)      # num_obs x rollouts x timesteps
    c_lane = np.max(np.maximum(0.0, -y_roll + y_lb), axis=1) + np.max(np.maximum(0.0, y_roll - y_ub), axis=1)
    return c_obs, c_lane


def var_index(alpha, n):
    """cvar_cost's linear-interpolation quantile position in float64: (lo, hi, lw, hw)"""
    q = alpha * (n - 1)
    lo, hi = math.floor(q), math.ceil(q)
    hw = q - lo
    return lo, hi, 1.0 - hw, hw


def mmd_sum_pairs(c, sigma):
    """S = sum_{i,j} exp(-|c_i - c_j| / sigma), the O(n^2) double sum"""
    c = np.asarray(c, np.float64)
    return float(np.sum(np.exp(-np.abs(c[:, None] - c[None, :]) / sigma)))


def mmd_sum_recurrence(c, sigma):
    """the same S = n + 2 sum_i P_i over the sorted costs, P_1 = 0, P_{i+1} = (P_i + 1) exp(-(v_{i+1} - v_i) / sigma)"""
    v = np.sort(np.asarray(c, np.float64))
    d = np.exp(-np.diff(v) / sigma)
    p, sp = 0.0, 0.0
    for x in d:
        p = (p + 1.0) * float(x)
        sp += p
    return v.size + 2.0 * sp


def risk_stats(c_obs, c_lane, alpha, sigma=None, ker_wt=1000.0, s_sum=mmd_sum_pairs):
    """dict p_coll, p_lane, mean_obs, var_obs, cvar_obs [, mmd_obs] of one plan's costs (c_lane None: p_lane = 0)"""
    c = np.asarray(c_obs, np.float64)
    n = c.size
    hit = lambda a: np.count_nonzero((a > 0) | np.isnan(a))
    out = dict(p_coll=hit(c) / n, p_lane=0.0 if c_lane is None else hit(np.asarray(c_lane, np.float64)) / n)
    if np.isnan(c).any():
        out.update(mean_obs=np.nan, var_obs=np.nan, cvar_obs=np.nan)
        if sigma is not None:
            out["mmd_obs"] = np.nan
        return out
    v = np.sort(c)
    lo, hi, lw, hw = var_index(alpha, n)
    var = v[lo] * lw + v[hi] * hw
    out.update(mean_obs=float(np.mean(c)), var_obs=float(var), cvar_obs=float(np.mean(c[c >= var])))
    if sigma is not None:
        E = float(np.sum(np.exp(-c / sigma)))
        out["mmd_obs"] = ker_wt * (s_sum(c, sigma) / (float(n) * n) - 2.0 * E / n)
    return out
