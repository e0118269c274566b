"""The CPU reference for cvar / saa / mmd_random above num_reduced 64 (tests/wide_oracle/oracle_wide.c through tests/wide_ref.py).

Up to 64 it must equal the frozen oracle bit for bit: the risk stage of the three costs under both noise models, and a small solve.  Above
64 there is no frozen oracle, so its cvar and saa are checked against a direct float32 NumPy restatement of the formulas (stable NaN-last
argsort, the quantile index q = alpha (n - 1), a sequential ascending-index tail sum) on vectors with many ties, all zeros, all positive
values and NaN."""
import numpy as np
import pytest

import wide_ref as W

f32 = np.float32
ST0 = np.array([0.0, 1.75, 5.0, 0.0, 0.0], f32)


@pytest.fixture(scope="module")
def O(built):
    from oracle import oracle
    oracle.set_threads(8)
    return oracle


@pytest.fixture(scope="module")
def wl(O, tmp_path_factory):
    return W.build_lib(tmp_path_factory.mktemp("wide_oracle"))


def _eq(a, b, what):
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert np.array_equal(a, b, equal_nan=True), f"{what}: got {a} want {b}"


def _controls(ora, rng, n):
    beq_x = np.array([0.0, 5.0, 0.0], f32); beq_y = np.array([1.75, 0.0, 0.0, 0.0], f32)
    acc, steer = [], []
    for _ in range(n):
        p = np.concatenate([rng.uniform(2, 25, 4), rng.normal(0, 3, 4)]).astype(f32)
        o = ora.project(p, beq_x, beq_y, 15.0, np.zeros(11, f32), np.zeros(11, f32), np.zeros(198, f32))
        acc.append(o["acc"]); steer.append(o["steer"])
    return np.stack(acc), np.stack(steer)


def _scene(O, ora):
    xo, yo, _ = ora.compute_obs_trajectories(*O.static_scene(2, 5))
    xo = xo.copy(); xo[0] = np.linspace(2, 60, 100); yo = yo.copy(); yo[0] = 1.75      # an obstacle on the path: rollouts collide
    return xo, yo


@pytest.mark.parametrize("noise", ["gaussian", "beta"])
@pytest.mark.parametrize("nr", [2, 5, 33, 64])
def test_wide_oracle_risk_equals_frozen_oracle(O, wl, nr, noise):
    args = (2, 0.3 if noise == "beta" else 0.1, 20, noise, 0.05, 0.01)
    ora = O.OracleCEM(nr, *args)
    wide = W.WideOracle(O, wl, nr, *args)
    acc, steer = _controls(ora, np.random.default_rng(100 + nr), 4)
    noise_t = ora.noise_tables(91, 2)
    for a, b in zip(noise_t[:4], wide.noise_tables(91, 2)[:4]):
        _eq(a, b, "noise tables")
    xo, yo = _scene(O, ora)
    collided = False
    for cost in ("cvar", "saa", "mmd_random"):
        for i in range(len(acc)):
            ref = ora.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo)
            got = wide.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo)
            for k in ("risk", "lane", "beta", "sigma", "red_cost"):
                _eq(got[k], ref[k], f"{cost} nr={nr} {noise} sample {i} {k}")
            collided |= bool((ref["red_cost"] > 0).any())
    assert collided


def test_wide_oracle_solve_equals_frozen_oracle(O, wl):
    args = (2, 0.3, 30, "beta", 0.02, 0.01)
    kw = dict(num_batch=24, maxiter_cem=2)
    ora = O.OracleCEM(33, *args, **kw)
    wide = W.WideOracle(O, wl, 33, *args, **kw)
    init_state, mean, cov, v_des = O.driver_inputs("static")
    (sc, idx) = O.static_episode(2, 3)
    xo, yo, _ = ora.compute_obs_trajectories(*sc)
    for cost in ("cvar", "saa"):
        ref = ora.solve(cost, idx, init_state, mean, cov, xo, yo, v_des)
        got = wide.solve(cost, idx, init_state, mean, cov, xo, yo, v_des)
        for k in ("cx", "cy", "cost_obs", "cost_lane", "sel"):
            _eq(got[k], ref[k], f"{cost} solve {k}")


# ---- above 64: the formulas restated in NumPy float32

def np_cvar(v, alpha=0.98):
    v = np.asarray(v, f32); n = v.size
    perm = np.argsort(v, kind="stable")                 # ascending, NaN last, ties in index order
    q = f32(alpha) * f32(n - 1)
    lo, hi = np.floor(q), np.ceil(q)
    hw = f32(q - lo); lw = f32(f32(1.0) - hw)
    ilo = min(max(int(lo), 0), n - 1); ihi = min(max(int(hi), 0), n - 1)
    var = f32(f32(v[perm[ilo]] * lw) + f32(v[perm[ihi]] * hw))
    s, cnt = f32(0.0), 0
    for x in v:
        if x >= var:
            s = f32(s + x); cnt += 1
    return f32(s / f32(cnt)) if cnt else f32(0.0)


def np_saa(v):
    v = np.asarray(v, f32)
    return f32(f32(np.count_nonzero(v > 0)) / f32(v.size))


def _vectors(n, rng):
    ties = rng.choice(np.array([0.0, 0.25, 0.5, 1.0], f32), n).astype(f32)
    mostly0 = np.where(rng.random(n) < 0.9, f32(0), rng.random(n).astype(f32)).astype(f32)
    pos = (rng.random(n) + f32(1e-3)).astype(f32)
    nan_top = pos.copy(); nan_top[rng.choice(n, 3, replace=False)] = np.nan
    nan_one = mostly0.copy(); nan_one[n // 2] = np.nan
    return dict(ties=ties, zeros=np.zeros(n, f32), mostly_zero=mostly0, positive=pos, nan3=nan_top, nan_one=nan_one,
                all_nan=np.full(n, np.nan, f32))


@pytest.mark.parametrize("n", [65, 96, 97, 100, 101, 128, 129, 256, 1001, 1023, 1024])
def test_wide_cvar_saa_match_numpy_restatement(wl, n):
    rng = np.random.default_rng(n)
    for name, v in _vectors(n, rng).items():
        _eq(W.cvar(wl, v), np_cvar(v), f"cvar n={n} {name}")
        _eq(W.saa(wl, v), np_saa(v), f"saa n={n} {name}")
    z = np.zeros(n, f32)
    assert W.cvar(wl, z) == 0 and W.saa(wl, z) == 0
    q = f32(0.98) * f32(n - 1)
    if n in (101, 1001):
        assert q == np.floor(q)                          # integer quantile index: lo == hi
    else:
        assert q != np.floor(q)
