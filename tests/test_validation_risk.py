"""Monte-Carlo risk statistics of the validation rollouts (DESIGN.md section 3 item 9): `risk_stats_batch`, `risk_stats`,
mpcmmd_validate_risk_host / mpcmmd_validate_threefry_risk_host / mpcmmd_risk_stats_host, `validation.py --risk`.
CPU: the restated definitions (tests/risk_oracle.py) against each other and the solver's cvar_cost formula, the Python layer's argument
checks and the command-line flags.  GPU: per-rollout costs against NumPy rollouts of the same perturbed controls, counts against the
counting entry points, the statistics kernel against the restatement on edge cases, chunking, invariants on solver plans, the CLI."""

import numpy as np
import pytest

import risk_oracle as RO
from test_validation import _cases, _fake_prob, _items
from test_validation_jax_rng import GROUPS, _group

STATS = ("p_coll", "p_lane", "mean_obs", "var_obs", "cvar_obs")


# ---- CPU -------------------------------------------------------------------------------------------------------------------------
def _rel(a, b):
    return abs(a - b) / max(abs(b), 1e-300)


@pytest.mark.parametrize("kind", ["random", "zeros", "ties"])
def test_oracle_mmd_recurrence_equals_double_sum(kind):
    """S = n + 2 sum P_i over the sorted costs equals the O(n^2) sum within 1e-12 relative: random costs, mostly exact zeros, ties"""
    rng = np.random.default_rng(7)
    for n in (1, 2, 3, 17, 500, 2000):
        if kind == "random":
            c = rng.random(n)
        elif kind == "zeros":
            c = np.where(rng.random(n) < 0.9, 0.0, rng.random(n))
        else:
            c = rng.choice([0.0, 0.25, 0.5, 0.5 + 1e-9], n)
        for sigma in (0.01, 0.1, 1.0, 10.0):
            assert _rel(RO.mmd_sum_recurrence(c, sigma), RO.mmd_sum_pairs(c, sigma)) <= 1e-12, (kind, n, sigma)


def _cvar_cost_var(v, alpha):
    """the VaR of the solver oracle's cvar_cost (oracle/oracle_mpc.c): stable argsort, q = alpha (nr - 1), floor / ceil clipped to the
    array, v[perm[lo]] lw + v[perm[hi]] hw -- restated in float64"""
    nr = len(v)
    perm = np.argsort(v, kind="stable")
    q = alpha * float(nr - 1)
    lo, hi = np.floor(q), np.ceil(q)
    hw = q - lo
    lw = 1.0 - hw
    ilo, ihi = min(max(int(lo), 0), nr - 1), min(max(int(hi), 0), nr - 1)
    return v[perm[ilo]] * lw + v[perm[ihi]] * hw


def test_oracle_var_is_cvar_cost_formula():
    """the restated VaR equals cvar_cost's formula on float32 costs widened to float64, bit for bit, and NumPy's linear quantile within
    2 ulp; CVaR is the mean of the costs at or above it"""
    rng = np.random.default_rng(3)
    for nr in (1, 2, 5, 8, 10, 40, 1000):
        for alpha in (0.0, 0.5, 0.9, 0.98, 1.0):
            v = np.maximum(rng.standard_normal(nr).astype(np.float32), np.float32(0)).astype(np.float64)
            got = RO.risk_stats(v, None, alpha)
            assert got["var_obs"] == _cvar_cost_var(v, alpha), (nr, alpha)
            want = np.quantile(v, alpha)
            assert abs(got["var_obs"] - want) <= 2 * np.spacing(max(abs(want), 1e-300)), (nr, alpha)
            assert got["cvar_obs"] == np.mean(v[v >= got["var_obs"]])


def _setup_cpu():
    g, _ = _cases()
    name = "S_beta_solve0"
    return _fake_prob("static", g[name + "_args"]), _items(g, [name])


def test_risk_argument_checks(built, monkeypatch):
    """alpha outside [0, 1], a bad sigma shape or value, rng="device", sigma with a Gaussian-kernel handle, bad costs: refused before
    the library is called"""
    from mpcmmd_b200 import binding as B, validation as V
    prob, item = _setup_cpu()

    def no_library():
        raise AssertionError("the library must not be called")
    monkeypatch.setattr(B, "load", no_library)
    run = lambda **kw: V.risk_stats_batch(prob, kw.pop("items", item), 50, 0.3, "beta", 4, device=0, **kw)
    for alpha in (-0.01, 1.01, float("nan")):
        with pytest.raises(ValueError, match="alpha"):
            run(alpha=alpha)
    for sigma in ([0.1, 0.2], np.zeros((1, 1)) + 0.1):
        with pytest.raises(ValueError, match="shape"):
            run(sigma=sigma)
    for sigma in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError, match="positive and finite"):
            run(sigma=sigma)
    with pytest.raises(ValueError, match="rng='host'"):
        run(rng="device")
    with pytest.raises(ValueError, match="'jax'"):
        run(rng="threefry")
    for n_roll in (0, 2.5, True):
        with pytest.raises(ValueError, match="n_roll"):
            run(n_roll=n_roll)
    prob.kernel = "gaussian"
    with pytest.raises(ValueError, match="Laplace"):
        run(sigma=0.01)
    run_stats = lambda c, **kw: V.risk_stats(c, device=0, **kw)
    for bad in (np.array([0.1, -0.2]), np.array([np.inf]), np.zeros(0), np.zeros((2, 2, 2))):
        with pytest.raises(ValueError, match="c_obs"):
            run_stats(bad)
    with pytest.raises(ValueError, match="c_lane"):
        run_stats(np.zeros(4), c_lane=np.zeros(5))
    with pytest.raises(ValueError, match="alpha"):
        run_stats(np.zeros(4), alpha=2.0)
    with pytest.raises(ValueError, match="shape"):
        run_stats(np.zeros((3, 4)), sigma=[0.1, 0.1])
    assert V.risk_stats_batch(prob, [], 50, 0.3, "beta", 4, device=0)["p_coll"].shape == (0,)


COMMON = ["--noises", "beta", "--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "4", "--num_prime", "50",
          "--acc_const_noise", "0.0", "--steer_const_noise", "0.0"]


def test_parser_risk_flags(built):
    from mpcmmd_b200 import validation as V
    a = V.build_parser().parse_args(COMMON)
    assert (a.risk, a.risk_alpha) == (False, 0.98)
    a = V.build_parser().parse_args(COMMON + ["--risk", "--risk_alpha", "0.9", "--rng", "jax"])
    assert (a.risk, a.risk_alpha, a.rng) == (True, 0.9, "jax")
    for bad in (["--risk_alpha", "1.5"], ["--risk_alpha", "-0.1"], ["--risk_alpha", "x"]):
        with pytest.raises(SystemExit):
            V.build_parser().parse_args(COMMON + bad)


def test_cli_risk_refuses_device_rng(built, tmp_path):
    """--risk with --rng device: the command line stops before anything is read, run_validation refuses it too"""
    from mpcmmd_b200 import validation as V
    argv = COMMON + ["--risk", "--rng", "device", "--root", str(tmp_path / "missing")]
    with pytest.raises(SystemExit):
        V.main(argv, variant="static")
    with pytest.raises(ValueError, match="--risk"):
        V.run_validation(V.build_parser().parse_args(argv), "static", log=lambda *a: None)


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _oracle_costs(V, prob, items, num_prime, num_obs, acc, steer):
    """NumPy rollouts (oracle_validation.rollouts) of the perturbed controls (n, n_roll, num_prime) and their costs, (n, n_roll) x2"""
    from oracle import oracle_validation as OV
    _, _, state0, xo, yo, static = V._inputs(prob, items, num_prime, num_obs)
    co, cl = np.empty(acc.shape[:2]), np.empty(acc.shape[:2])
    for i in range(len(items)):
        xr, yr = OV.rollouts(acc[i], steer[i], state0[i], prob.t, prob.wheel_base)
        co[i], cl[i] = RO.rollout_costs(xr, yr, xo[i], yo[i], num_prime, prob.a_obs, prob.b_obs, prob.y_lb, prob.y_ub, static)
    return co, cl, static


def _check_costs(got_o, got_l, want_o, want_l, static, tag):
    """static c_obs within 1 float32 ulp, everything else within 1e-12 relative; no oracle cost within 1e-9 of 0, so that the hit
    indicators cannot flip; then the probabilities are identical"""
    for w in (want_o, want_l):
        assert not np.any((w != 0) & (np.abs(w) < 1e-9)), tag
    if static:
        ulp = np.spacing(np.abs(want_o).astype(np.float32)).astype(np.float64)
        assert np.all(np.abs(got_o - want_o) <= ulp), (tag, np.max(np.abs(got_o - want_o) / ulp))
    else:
        assert np.allclose(got_o, want_o, rtol=1e-12, atol=0), tag
    assert np.allclose(got_l, want_l, rtol=1e-12, atol=0), tag
    assert np.array_equal(got_o > 0, want_o > 0) and np.array_equal(got_l > 0, want_l > 0), tag


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["S_beta", "S_gauss", "D_gauss", "D_beta"])
def test_host_draws_costs_match_numpy_rollouts(built, group):
    """golden validation cases, NumPy's noise, 1000 rollouts: c_obs / c_lane of mpcmmd_validate_risk_host against the oracle's rollouts of
    the same perturbed controls; p_coll / p_lane identical to the oracle's; counts identical to compute_stats_batch's"""
    _need_gpu()
    from mpcmmd_b200 import validation as V
    g, _ = _cases()
    names, prob, num_obs, noise_level, num_prime, noise = _group(g, group)
    items = _items(g, names)
    got = V.risk_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, want_rollout_costs=True, device=0)
    acc_p, steer_p, _, _, _, _ = V._inputs(prob, items, num_prime, num_obs)
    drawn = [V.perturbed_controls(prob, acc_p[i], steer_p[i], noise_level, num_prime, noise, it["key"]) for i, it in enumerate(items)]
    acc, steer = np.stack([d[0] for d in drawn]), np.stack([d[1] for d in drawn])
    want_o, want_l, static = _oracle_costs(V, prob, items, num_prime, num_obs, acc, steer)
    _check_costs(got["c_obs"], got["c_lane"], want_o, want_l, static, group)
    for i in range(len(items)):
        o = RO.risk_stats(want_o[i], want_l[i], 0.98)
        assert got["p_coll"][i] == o["p_coll"] and got["p_lane"][i] == o["p_lane"], (group, i)
    count, lane = V.compute_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, device=0)
    assert np.array_equal(got["count"], count) and np.array_equal(got["count_lane"], lane)


@pytest.mark.gpu
@pytest.mark.parametrize("n_roll", [257, 4099])
def test_counter_noise_costs_match_numpy_rollouts(built, n_roll):
    """counter-based noise at n_roll not a multiple of the block: the per-rollout costs against NumPy rollouts of the perturbed controls
    threefry_stats_batch returns for the same seeds; counts identical to threefry_stats_batch's"""
    _need_gpu()
    from mpcmmd_b200 import validation as V
    g, _ = _cases()
    for group in GROUPS:
        names, prob, num_obs, noise_level, num_prime, noise = _group(g, group)
        items = _items(g, names)
        got = V.risk_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, n_roll=n_roll, rng="jax", want_rollout_costs=True, device=0)
        count, lane, acc, steer = V.threefry_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, want_draws=True, device=0, n_roll=n_roll)
        want_o, want_l, static = _oracle_costs(V, prob, items, num_prime, num_obs, acc, steer)
        _check_costs(got["c_obs"], got["c_lane"], want_o, want_l, static, (group, n_roll))
        assert np.array_equal(got["count"], count) and np.array_equal(got["count_lane"], lane), (group, n_roll)
        for i in range(len(items)):
            o = RO.risk_stats(want_o[i], want_l[i], 0.98)
            assert got["p_coll"][i] == o["p_coll"] and got["p_lane"][i] == o["p_lane"], (group, i)


def _edge_sets(rng):
    """(label, c_obs, c_lane) edge cases of the statistics kernel"""
    out = []
    for n in (1, 2, 3, 255, 256, 257, 100007):
        lane = np.where(rng.random(n) < 0.2, rng.random(n) * 3, 0.0)
        out.append(("zeros", np.zeros(n), lane))
        out.append(("equal", np.full(n, 0.3712), lane))
        one = np.zeros(n); one[rng.integers(n)] = 0.625
        out.append(("one", one, lane))
        out.append(("all_nonzero", rng.random(n) * 0.9 + 1e-3, lane))
        out.append(("mixed", np.where(rng.random(n) < 0.8, 0.0, rng.random(n)), lane))
        out.append(("ties", rng.choice([0.0, 0.125, 0.5, 0.5 + 2 ** -40], n), lane))
        for pos in sorted({0, n // 2, n - 1}):
            c = rng.random(n) * 0.5
            c[pos] = np.nan
            out.append(("nan@%d" % pos, c, lane))
    return out


def _compare_stats(got, want, i, label):
    for k in ("p_coll", "p_lane", "var_obs"):
        g_, w_ = np.float64(got[k][i]), np.float64(want[k])
        assert g_.tobytes() == w_.tobytes() or (np.isnan(g_) and np.isnan(w_)), (label, k, g_, w_)
    for k in ("mean_obs", "cvar_obs") + (("mmd_obs",) if "mmd_obs" in want else ()):
        g_, w_ = float(got[k][i]), float(want[k])
        if np.isnan(w_):
            assert np.isnan(g_), (label, k)
        else:
            assert abs(g_ - w_) <= 1e-12 * max(abs(w_), 1e-300), (label, k, g_, w_)


@pytest.mark.gpu
def test_stats_kernel_edge_cases(built):
    """mpcmmd_risk_stats_host against the restatement: all zeros, all equal, one nonzero, every value nonzero, ties, NaN at the first /
    a middle / the last position, n in {1, 2, 3, 255, 256, 257, 10^5 + 7}, alpha in {0, 0.5, 0.98, 1} and one with alpha (n - 1) an
    integer.  VaR and the probabilities bit for bit, mean / CVaR / MMD within 1e-12 relative (MMD against the O(n^2) sum up to
    n = 4096, the recurrence above); a second call gives the same bits"""
    _need_gpu()
    from mpcmmd_b200 import validation as V
    rng = np.random.default_rng(11)
    sets = _edge_sets(rng)
    for n in sorted({len(c) for _, c, _ in sets}):
        group = [(l, c, cl) for l, c, cl in sets if len(c) == n]
        co = np.stack([c for _, c, _ in group]); cl = np.stack([x for _, _, x in group])
        sigma = np.array([0.01, 0.1, 1.0] * len(group))[:len(group)]
        for alpha in (0.0, 0.5, 0.98, 1.0) + ((0.75,) if n > 1 and (0.75 * (n - 1)).is_integer() else (0.5 if n == 1 else 1.0 / (n - 1),)):
            got = V.risk_stats(co, cl, alpha=alpha, sigma=sigma, ker_wt=1000.0, device=0)
            again = V.risk_stats(co, cl, alpha=alpha, sigma=sigma, ker_wt=1000.0, device=0)
            for k in got:
                assert np.asarray(got[k]).tobytes() == np.asarray(again[k]).tobytes(), (n, alpha, k)
            for i, (label, c, x) in enumerate(group):
                s_sum = RO.mmd_sum_pairs if n <= 4096 else RO.mmd_sum_recurrence
                want = RO.risk_stats(c, x, alpha, sigma=sigma[i], ker_wt=1000.0, s_sum=s_sum)
                _compare_stats(got, want, i, (label, n, alpha))
    one = V.risk_stats(np.array([0.0, 0.5, 0.25]), alpha=0.5)                  # a single set, no c_lane, no sigma
    assert float(one["var_obs"]) == 0.25 and float(one["p_lane"]) == 0.0 and "mmd_obs" not in one


@pytest.mark.gpu
def test_chunked_call_equals_separate_calls(built):
    """700 plans x 10^5 rollouts of counter-based noise (1.1 GB of per-rollout costs, beyond the 1 GiB scratch: two chunks) give the
    statistics, bit for bit, of the same plans validated in separate calls, on both sides of the chunk boundary"""
    _need_gpu()
    from mpcmmd_b200 import validation as V
    g, _ = _cases()
    names, prob, num_obs, noise_level, num_prime, noise = _group(g, "S_beta")
    base = _items(g, names[:1])[0]
    items = [dict(base, key=k) for k in range(700)]
    n_roll = 100000
    assert len(items) * n_roll * 16 > 2 ** 30
    kw = dict(n_roll=n_roll, rng="jax", sigma=0.05, device=0)
    full = V.risk_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, **kw)
    assert np.any(full["p_coll"] > 0)
    for lo, hi in ((0, 3), (668, 674), (697, 700)):
        part = V.risk_stats_batch(prob, items[lo:hi], num_prime, noise_level, noise, num_obs, **kw)
        for k in STATS + ("mmd_obs", "count", "count_lane"):
            assert full[k][lo:hi].tobytes() == part[k].tobytes(), (k, lo, hi)


@pytest.mark.gpu
def test_invariants_on_solver_plans(built):
    """cvar and mmd_opt plans of 12 static episodes at 2 x 10^4 rollouts: count <= p_coll n_roll, count_lane <= 2 p_lane n_roll, the
    moments ordered mean <= CVaR, VaR <= CVaR, and the MMD of the solver's own bandwidth finite"""
    _need_gpu()
    from mpcmmd_b200 import CEM, scenes, validation as V
    prob = CEM(5, 4, 0.3, 50, "beta", 0.0, 0.0, variant="static", max_episodes=12)
    eps = list(range(12))
    batch = scenes.static_batch(prob, eps)
    init_state = scenes.driver_inputs("static")[0]
    n_roll = 20000
    for cost in ("cvar", "mmd_opt"):
        out = prob.solve_batch(cost, **batch)
        items = []
        for k in eps:
            (x, y, vx, vy, _), _ = scenes.static_scene(4, k)
            items.append(dict(cx=out["cx"][k].astype(np.float64), cy=out["cy"][k].astype(np.float64), init_state=init_state.astype(np.float64),
                              key=k, x_obs=x.astype(np.float64), y_obs=y.astype(np.float64), vx_obs=vx, vy_obs=vy))
        sigma = np.asarray(out["sigma"], np.float64) if cost == "mmd_opt" else None
        for rng in ("host", "jax"):
            r = V.risk_stats_batch(prob, items, 50, 0.3, "beta", 4, n_roll=n_roll, rng=rng, sigma=sigma, device=0)
            hits, hits_lane = np.rint(r["p_coll"] * n_roll), np.rint(r["p_lane"] * n_roll)
            assert np.all(r["count"] <= hits) and np.all(r["count_lane"] <= 2 * hits_lane), (cost, rng)
            tol = 1e-12 * np.abs(r["cvar_obs"])
            assert np.all(r["mean_obs"] <= r["cvar_obs"] + tol) and np.all(r["var_obs"] <= r["cvar_obs"] + tol), (cost, rng)
            if sigma is not None:
                assert np.all(np.isfinite(r["mmd_obs"])), (cost, rng)


@pytest.mark.gpu
def test_cli_risk_writes_extra_keys(built, tmp_path):
    """validation.py --risk --rng jax --num_rollouts 2000: the stats file has the reference keys, rng / num_rollouts, risk_alpha and the
    ten risk arrays with the lengths of the coll_* arrays, and its counts are those of the run without --risk"""
    _need_gpu()
    from mpcmmd_b200 import driver, validation as V
    common = COMMON + ["--root", str(tmp_path / "data")]
    driver.run_sweep(driver.build_parser().parse_args(common + ["--costs", "cvar", "mmd_opt", "--num_configs", "5"]), log=lambda *a: None)
    run = lambda sub, extra: np.load(V.run_validation(V.build_parser().parse_args(common + ["--stats_root", str(tmp_path / sub), "--rng", "jax",
                                                                                           "--num_rollouts", "2000"] + extra), "static",
                                                      log=lambda *a: None)[0])
    st, plain = run("risk", ["--risk", "--risk_alpha", "0.9"]), run("plain", [])
    risk_keys = {k + s for k in STATS for s in ("_cvar", "_mmd_opt")}
    assert set(st.files) == set(plain.files) | risk_keys | {"risk_alpha"}
    assert float(st["risk_alpha"]) == 0.9
    for s in ("_cvar", "_mmd_opt"):
        m = st["coll" + s].shape
        for k in STATS:
            assert st[k + s].shape == m, k + s
        assert np.all(st["coll" + s] <= np.rint(st["p_coll" + s] * 2000))
    for k in plain.files:
        assert np.array_equal(st[k], plain[k]), k
