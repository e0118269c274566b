"""Monte-Carlo validation with counter-based noise (`compute_stats_batch(..., rng="jax")`, csrc/k_validate_jax.cuh; DESIGN.md section 3
item 7).  The stream definition is restated on the CPU from the pinned oracle's JAX primitives (oracle.prng_key / split / beta / normal)
plus validation.perturbed_controls' float64 expressions.  CPU: the restatement against JAX itself when JAX is importable, the Python
layer's argument checks and the command-line flags.  GPU: the kernel's perturbed controls against the restatement bit for bit, its counts
against mpcmmd_validate_host on the restated controls, and its counts against NumPy-noise counts in distribution."""
import ctypes as C

import numpy as np
import pytest

from test_validation import _cases, _fake_prob, _items

REF_KEYS = {"coll_cvar", "coll_cvar_lane", "coll_mmd_opt", "coll_mmd_opt_lane", "coll_mmd_random", "coll_mmd_random_lane"}
GROUPS = ["S_beta", "S_gauss", "D_gauss", "D_beta"]


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def restated_draws(prob, acc, steer, num_prime, noise, key, n_roll):
    """the float32 draws of item 1 for one trajectory, each (n_roll, num_prime): {"acc", "steer", "z"} -- Beta draws for beta noise,
    standard normals for Gaussian noise -- from the oracle's restatement of the JAX 0.3.23 PRNG"""
    from oracle import oracle as O
    k_acc, k_steer, k_z = (tuple(int(v) for v in row) for row in O.split(O.prng_key(key), 3))
    n = n_roll * num_prime
    shape = lambda p: np.ascontiguousarray(np.broadcast_to(np.asarray(p, np.float64).astype(np.float32), (n_roll, num_prime)))
    if noise == "beta":
        d = dict(acc=O.beta(k_acc, shape(prob.beta_a * np.abs(acc)), shape(prob.beta_b * np.abs(acc))),
                 steer=O.beta(k_steer, shape(prob.beta_a * np.abs(steer) + 1e-5), shape(prob.beta_b * np.abs(steer) + 1e-5)))
    else:
        d = dict(acc=O.normal(k_acc, n), steer=O.normal(k_steer, n))
    d["z"] = O.normal(k_z, n)
    return {k: v.reshape(n_roll, num_prime) for k, v in d.items()}


def restated_controls(prob, acc, steer, noise_level, num_prime, noise, key, n_roll):
    """the perturbed controls of item 1: the draws widened to float64, then perturbed_controls' expressions"""
    d = {k: v.astype(np.float64) for k, v in restated_draws(prob, acc, steer, num_prime, noise, key, n_roll).items()}
    if noise == "gaussian":
        acc_pert = noise_level * np.abs(acc) * d["acc"]
        steer_pert = noise_level * np.abs(steer) * d["steer"]
    else:
        acc_pert = noise_level * (2 * d["acc"] - 1)
        steer_pert = prob.cem_helper.K_steer * noise_level * (2 * d["steer"] - 1)
    return acc + acc_pert + prob.acc_const_noise * d["z"], steer + steer_pert + prob.steer_const_noise * d["z"]


def _group(g, group):
    """(names, fake prob, num_obs, noise_level, num_prime, noise) of one group of golden cases"""
    names = [n for n in _cases()[1] if n.startswith(group)]
    args = g[names[0] + "_args"]
    prob = _fake_prob("static" if group.startswith("S_") else "dynamic", args)
    return names, prob, int(args[1]), float(args[2]), int(args[3]), ("gaussian", "beta")[int(args[4])]


def _restated(V, prob, items, num_prime, num_obs, noise_level, noise, n_roll):
    """restated_controls of every item: (n, n_roll, num_prime) x2"""
    acc_p, steer_p, _, _, _, _ = V._inputs(prob, items, num_prime, num_obs)
    a = np.empty((len(items), n_roll, num_prime)); s = np.empty_like(a)
    for i, it in enumerate(items):
        a[i], s[i] = restated_controls(prob, acc_p[i], steer_p[i], noise_level, num_prime, noise, it["key"], n_roll)
    return a, s


# ---- CPU -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("noise", ["beta", "gaussian"])
def test_restatement_matches_jax(built, noise):
    """the restated draws are jax.random.beta / normal of split(PRNGKey(k), 3), element for element (needs JAX 0.3.23)"""
    jax = pytest.importorskip("jax")
    if "jax_shim" in getattr(jax, "__file__", ""):
        pytest.skip("the NumPy stand-in for JAX is built on the oracle itself")
    from jax import random
    from mpcmmd_b200 import validation as V
    g, _ = _cases()
    name = "S_beta_solve0" if noise == "beta" else "S_gauss_solve0"
    prob = _fake_prob("static", g[name + "_args"])
    acc, steer = V.compute_controls(prob, g[name + "_cx"], g[name + "_cy"])
    acc, steer = acc[:50], steer[:50]
    for key, n_roll in ((0, 3), (12345, 257), (2 ** 32 - 1, 10)):
        want = restated_draws(prob, acc, steer, 50, noise, key, n_roll)
        k_acc, k_steer, k_z = random.split(random.PRNGKey(key), 3)
        if noise == "beta":
            f32 = lambda p: np.broadcast_to(np.asarray(p, np.float64).astype(np.float32), (n_roll, 50))
            got = dict(acc=random.beta(k_acc, f32(prob.beta_a * np.abs(acc)), f32(prob.beta_b * np.abs(acc)), (n_roll, 50)),
                       steer=random.beta(k_steer, f32(prob.beta_a * np.abs(steer) + 1e-5), f32(prob.beta_b * np.abs(steer) + 1e-5), (n_roll, 50)))
        else:
            got = dict(acc=random.normal(k_acc, (n_roll, 50)), steer=random.normal(k_steer, (n_roll, 50)))
        got["z"] = random.normal(k_z, (n_roll, 50))
        for k in want:
            assert np.array_equal(np.asarray(got[k]).view(np.uint32), want[k].view(np.uint32)), (key, n_roll, k)


def test_restatement_zero_shape_gives_nan_at_last_knot(built):
    """beta noise at num_prime = 100: acc[99] == 0 makes both Beta shapes 0, and the restated sampler returns NaN there (no argument
    check, as JAX makes none); every other draw of the trajectory is finite"""
    from mpcmmd_b200 import validation as V
    g, _ = _cases()
    name = "S_beta_solve0"
    prob = _fake_prob("static", g[name + "_args"])
    acc, steer = V.compute_controls(prob, g[name + "_cx"], g[name + "_cy"])
    assert acc[99] == 0.0
    a, s = restated_controls(prob, acc[:100], steer[:100], 0.3, 100, "beta", int(g[name + "_args"][7]), 64)
    assert np.isnan(a[:, 99]).all() and np.isfinite(a[:, :99]).all() and np.isfinite(s).all()


def test_jax_rng_argument_checks(built, monkeypatch):
    """seeds in np.random.seed's range, n_roll >= 1 with n_roll * num_prime < 2**31, rng spelled right, no rollouts; no Beta shape
    check (num_prime = 100 reaches the library).  All refused before the library is called."""
    from mpcmmd_b200 import binding as B, validation as V
    g, _ = _cases()
    name = "S_beta_solve0"
    args = g[name + "_args"]
    prob = _fake_prob("static", args)
    item = _items(g, [name])

    def no_library():
        raise AssertionError("the library must not be called")
    monkeypatch.setattr(B, "load", no_library)
    run = lambda items=item, **kw: V.compute_stats_batch(prob, items, kw.pop("num_prime", 50), 0.3, "beta", 4, device=0, **kw)
    for key in (2 ** 32, -1):
        with pytest.raises(ValueError, match="Seed must be between"):
            run([dict(item[0], key=key)], rng="jax")
    for n_roll in (0, -5, 2.5, True):
        with pytest.raises(ValueError, match="n_roll"):
            run(rng="jax", n_roll=n_roll)
    with pytest.raises(ValueError, match="2\\*\\*31"):
        run(rng="jax", n_roll=2 ** 31 // 50 + 1)
    with pytest.raises(ValueError, match="rng='host'"):
        run(rng="jax", want_rollouts=True)
    with pytest.raises(ValueError, match="'jax'"):
        run(rng="threefry")
    with pytest.raises(ValueError, match="noise"):
        V.threefry_stats_batch(prob, item, 50, 0.3, "uniform", 4, device=0)
    with pytest.raises(AssertionError, match="library"):                # num_prime = 100, acc[99] == 0: no "a <= 0"
        run(rng="jax", num_prime=100)
    assert [len(x) for x in V.threefry_stats_batch(prob, [], 50, 0.3, "beta", 4, device=0)] == [0, 0]


def test_parser_jax_rng_and_num_rollouts(built):
    from mpcmmd_b200 import validation as V
    common = ["--noises", "beta", "--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "4", "--num_prime", "50",
              "--acc_const_noise", "0.0", "--steer_const_noise", "0.0"]
    a = V.build_parser().parse_args(common)
    assert (a.rng, a.num_rollouts) == ("host", 1000)
    a = V.build_parser().parse_args(common + ["--rng", "jax", "--num_rollouts", "100000"])
    assert (a.rng, a.num_rollouts) == ("jax", 100000)
    assert V.build_parser().parse_args(common + ["--rng", "device", "--num_rollouts", "1"]).num_rollouts == 1
    for bad in (["--num_rollouts", "0"], ["--num_rollouts", "-3"], ["--num_rollouts", "1e5"], ["--rng", "numpy"]):
        with pytest.raises(SystemExit):
            V.build_parser().parse_args(common + bad)


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _validate_host(V, B, prob, items, num_prime, num_obs, acc, steer):
    """mpcmmd_validate_host's counts on given perturbed controls (n, n_roll, num_prime)"""
    _, _, state0, xo, yo, static = V._inputs(prob, items, num_prime, num_obs)
    n, n_roll = acc.shape[:2]
    count, lane = np.zeros(n, np.int32), np.zeros(n, np.int32)
    B.check(B.load().mpcmmd_validate_host(0, n, n_roll, num_prime, num_obs, 1 if static else 0, *V._geometry(prob), _p(np.ascontiguousarray(acc)),
                                          _p(np.ascontiguousarray(steer)), _p(state0), _p(xo), _p(yo), _p(count), _p(lane), None, None))
    return count, lane


@pytest.mark.gpu
@pytest.mark.parametrize("n_roll", [1000, 1, 255, 257, 4099])
def test_jax_rng_matches_restatement_on_golden_cases(built, n_roll):
    """all 12 golden cases (both variants, both noises): the kernel's perturbed controls are the restatement's bit for bit, and its
    counts are mpcmmd_validate_host's on the restated controls; n_roll straddles the 256-rollout chunks"""
    _need_gpu()
    from mpcmmd_b200 import binding as B, validation as V
    g, _ = _cases()
    for group in GROUPS:
        names, prob, num_obs, noise_level, num_prime, noise = _group(g, group)
        items = _items(g, names)
        count, lane, a_d, s_d = V.threefry_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, want_draws=True, device=0, n_roll=n_roll)
        a_r, s_r = _restated(V, prob, items, num_prime, num_obs, noise_level, noise, n_roll)
        assert np.array_equal(a_d, a_r) and np.array_equal(s_d, s_r), (group, n_roll)
        hc, hl = _validate_host(V, B, prob, items, num_prime, num_obs, a_r, s_r)
        assert np.array_equal(count, hc) and np.array_equal(lane, hl), (group, n_roll, count, hc, lane, hl)
        c2, l2 = V.compute_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, device=0, n_roll=n_roll, rng="jax")
        assert np.array_equal(count, c2) and np.array_equal(lane, l2)


@pytest.mark.gpu
def test_jax_rng_beta_at_num_prime_100(built):
    """beta noise at num_prime = 100, which the NumPy modes refuse (acc[99] == 0): the NaN draws of the last knot reach only the
    discarded final state, and the counts equal those of the restated controls"""
    _need_gpu()
    from mpcmmd_b200 import binding as B, validation as V
    g, _ = _cases()
    names, prob, num_obs, noise_level, _, noise = _group(g, "S_beta")
    items = _items(g, names)
    count, lane, a_d, s_d = V.threefry_stats_batch(prob, items, 100, noise_level, noise, num_obs, want_draws=True, device=0, n_roll=1000)
    a_r, s_r = _restated(V, prob, items, 100, num_obs, noise_level, noise, 1000)
    assert np.array_equal(a_d, a_r, equal_nan=True) and np.array_equal(s_d, s_r) and np.isnan(a_d[:, :, 99]).all()
    hc, hl = _validate_host(V, B, prob, items, 100, num_obs, a_r, s_r)
    assert np.array_equal(count, hc) and np.array_equal(lane, hl)


@pytest.mark.gpu
def test_jax_rng_agrees_with_numpy_noise_in_distribution(built):
    """at 2 x 10^5 rollouts, count / n_roll and count_lane / n_roll of rng="jax" and rng="host" (NumPy's stream) agree within
    5 standard deviations, on the golden plans with nonzero collision counts (four beta, two Gaussian)"""
    _need_gpu()
    from mpcmmd_b200 import validation as V
    n = 200000
    g, _ = _cases()
    plans = {"S_beta": ["S_beta_solve0", "S_beta_solve3"], "D_beta": ["D_beta_solve0", "D_beta_solve2"],
             "S_gauss": ["S_gauss_solve0"], "D_gauss": ["D_gauss_solve0"]}
    for group, names in plans.items():
        _, prob, num_obs, noise_level, num_prime, noise = _group(g, group)
        items = _items(g, names)
        got = {rng: V.compute_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, device=0, n_roll=n, rng=rng) for rng in ("jax", "host")}
        for i, name in enumerate(names):
            cj, ch = int(got["jax"][0][i]), int(got["host"][0][i])
            assert ch > 0, name
            p = (cj + ch) / (2.0 * n)                                      # a max over (obstacle, t) of binomial counts, <= n
            sd = max(np.sqrt(2 * p * (1 - p) / n), 1.0 / n)
            assert abs(cj - ch) / n <= 5 * sd, (name, "count", cj, ch, sd * n)
            lj, lh = int(got["jax"][1][i]), int(got["host"][1][i])
            q = (lj + lh) / (4.0 * n)                                      # the sum of two such maxima, <= 2n: sd <= 2 sqrt(n q (1 - q))
            sd = max(2 * np.sqrt(2 * q * (1 - q) / n), 1.0 / n)
            assert abs(lj - lh) / n <= 5 * sd, (name, "lane", lj, lh, sd * n)
            print("%s: count %d / %d (jax / NumPy), lane %d / %d of %d rollouts" % (name, cj, ch, lj, lh, n))


@pytest.mark.gpu
def test_jax_rng_beta_draws_have_beta_moments(built):
    """at 10^5 rollouts the Beta draws recovered from the perturbed controls have, per knot, the mean a / (a + b) and the variance
    ab / ((a + b)^2 (a + b + 1)) of their f32 shapes within 5 standard errors"""
    _need_gpu()
    from mpcmmd_b200 import validation as V
    g, _ = _cases()
    names, prob, num_obs, noise_level, num_prime, noise = _group(g, "S_beta")
    assert prob.acc_const_noise == 0.0 and prob.steer_const_noise == 0.0          # the controls carry the Beta draws alone
    items = _items(g, names[:1])
    n = 100000
    _, _, a_d, s_d = V.threefry_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, want_draws=True, device=0, n_roll=n)
    acc_p, steer_p, _, _, _, _ = V._inputs(prob, items, num_prime, num_obs)
    ks = prob.cem_helper.K_steer * noise_level
    for b, a_sh, b_sh in ((((a_d[0] - acc_p[0]) / noise_level + 1) / 2, prob.beta_a * np.abs(acc_p[0]), prob.beta_b * np.abs(acc_p[0])),
                          (((s_d[0] - steer_p[0]) / ks + 1) / 2, prob.beta_a * np.abs(steer_p[0]) + 1e-5, prob.beta_b * np.abs(steer_p[0]) + 1e-5)):
        a_sh, b_sh = a_sh.astype(np.float32).astype(np.float64), b_sh.astype(np.float32).astype(np.float64)
        mu = a_sh / (a_sh + b_sh)
        var = a_sh * b_sh / ((a_sh + b_sh) ** 2 * (a_sh + b_sh + 1))
        m = b.mean(axis=0)
        dev = b - m
        s2 = (dev ** 2).mean(axis=0)
        m4 = (dev ** 4).mean(axis=0)
        assert np.all(np.abs(m - mu) <= 5 * np.sqrt(var / n)), np.max(np.abs(m - mu) / np.sqrt(var / n))
        assert np.all(np.abs(s2 - var) <= 5 * np.sqrt((m4 - s2 ** 2) / n)), np.max(np.abs(s2 - var) / np.sqrt((m4 - s2 ** 2) / n))


@pytest.mark.gpu
def test_run_validation_jax_rng_writes_tagged_stats(built, tmp_path):
    """the README workflow (5 static episodes, cvar + mmd_opt) with --rng jax --num_rollouts 5000: the six reference keys with one
    entry per matched pair, plus rng and num_rollouts; the host draws at a non-default rollout count are tagged too"""
    _need_gpu()
    from mpcmmd_b200 import driver, validation as V
    common = ["--noises", "beta", "--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "4", "--num_prime", "50",
              "--acc_const_noise", "0.0", "--steer_const_noise", "0.0", "--root", str(tmp_path / "data")]
    driver.run_sweep(driver.build_parser().parse_args(common + ["--costs", "cvar", "mmd_opt", "--num_configs", "5"]), log=lambda *a: None)
    d_c = V._load(str(tmp_path / "data"), "beta", 0.3, 50, "cvar", 5, 4)
    d_o = V._load(str(tmp_path / "data"), "beta", 0.3, 50, "mmd_opt", 5, 4)
    m = len(V.matched_pairs(d_c, d_o, 4))
    assert m >= 1
    for rng, n_roll in (("jax", 5000), ("host", 1500)):
        args = V.build_parser().parse_args(common + ["--stats_root", str(tmp_path / rng), "--rng", rng, "--num_rollouts", str(n_roll)])
        path, = V.run_validation(args, "static", log=lambda *a: None)
        st = np.load(path)
        assert set(st.files) == REF_KEYS | {"rng", "num_rollouts"}
        assert str(st["rng"]) == rng and int(st["num_rollouts"]) == n_roll
        for k in ("coll_cvar", "coll_cvar_lane", "coll_mmd_opt", "coll_mmd_opt_lane"):
            assert st[k].shape == (m,) and np.all(st[k] >= 0) and np.all(st[k] <= 2 * n_roll), k
        assert st["coll_mmd_random"].shape == (0,)
