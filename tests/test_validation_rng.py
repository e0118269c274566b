"""Monte-Carlo validation with the noise drawn on the device (`compute_stats_batch(..., rng="device")`, csrc/dnprng.cuh,
csrc/k_validate_noise.cuh).  CPU: the C restatement of NumPy's legacy stream (tests/nprng/oracle_nprng.h, the contract of DESIGN.md
section 3 item 6) against NumPy itself, bit for bit, and the Python layer's argument checks.  GPU: the device streams against the host
draws (identical stream consumption, values within CUDA's libm rounding) and the counts against the host path and the golden vectors."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from test_validation import _case_inputs, _cases, _fake_prob, _items

HERE = os.path.dirname(os.path.abspath(__file__))
NPRNG = os.path.join(HERE, "nprng")
WORDS = 628
UINT32_MAX = 2 ** 32 - 1


@pytest.fixture(scope="session")
def nprng(tmp_path_factory):
    """the C restatement built with the oracle's arithmetic flags (glibc's pow / log / exp, as NumPy's)"""
    out = str(tmp_path_factory.mktemp("nprng") / "liboracle_nprng.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-Wall",
                           os.path.join(NPRNG, "oracle_nprng.c"), "-o", out, "-lm"])
    lib = C.CDLL(out)
    V = C.c_void_p
    lib.oracle_npr_seed.argtypes = [C.c_uint32, V]
    lib.oracle_npr_draw.argtypes = [V, C.c_int, C.c_int, V, V, V]
    lib.oracle_npr_perturbed.argtypes = [C.c_uint32, C.c_int, C.c_int, C.c_int, V, V] + [C.c_double] * 6 + [V, V, V]
    return lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def numpy_state():
    """np.random.get_state() in the 628-word layout of mpcmmd_validate_seeded_host's state_out"""
    _, key, pos, has_gauss, gauss = np.random.get_state()
    w = np.empty(WORDS, np.uint32)
    w[:624] = key; w[624] = pos; w[625] = has_gauss
    w[626:] = np.array([gauss], np.float64).view(np.uint32)
    return w


def _draw(lib, state, kind, n, p1=None, p2=None):
    out = np.empty(n)
    p1 = None if p1 is None else np.ascontiguousarray(np.broadcast_to(np.float64(p1), (n,)))
    p2 = None if p2 is None else np.ascontiguousarray(np.broadcast_to(np.float64(p2), (n,)))
    lib.oracle_npr_draw(_p(state), kind, n, _p(p1), _p(p2), _p(out))
    return out


def oracle_perturbed(lib, prob, acc, steer, noise_level, num_prime, noise, key, n_roll=1000):
    a, s, st = np.empty((n_roll, num_prime)), np.empty((n_roll, num_prime)), np.empty(WORDS, np.uint32)
    acc, steer = np.ascontiguousarray(acc, np.float64), np.ascontiguousarray(steer, np.float64)
    lib.oracle_npr_perturbed(key, 1 if noise == "beta" else 0, n_roll, num_prime, _p(acc), _p(steer), noise_level, prob.cem_helper.K_steer,
                             float(prob.beta_a), float(prob.beta_b), prob.acc_const_noise, prob.steer_const_noise, _p(a), _p(s), _p(st))
    return a, s, st


# ---- CPU -------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 3, 17, UINT32_MAX])
def test_oracle_primitives_match_numpy(nprng, seed):
    """every primitive of the restatement draws NumPy's values bit for bit and leaves np.random.get_state() as NumPy does, over one
    continuing stream: odd-length normal draws carry the one-value cache into the next call; the gamma shapes reach shape < 1
    (both branches), == 1 and > 1; the beta grid reaches Johnk, its log-space branch ((1e-5, 1e-5), (2e-15, 5e-15)) and Ga / (Ga + Gb)"""
    np.random.seed(seed)
    st = np.empty(WORDS, np.uint32)
    nprng.oracle_npr_seed(seed, _p(st))
    assert np.array_equal(st, numpy_state())
    calls = [(0, 7, None, None, lambda: np.random.random_sample(7)),
             (1, 5, None, None, lambda: np.random.standard_normal(5)),
             (2, 6, None, None, lambda: np.random.standard_exponential(6)),
             (1, 3, None, None, lambda: np.random.standard_normal(3))]
    for shape in (1e-3, 0.4, 1.0, 1.7, 5.0):
        calls.append((3, 9, shape, None, lambda sh=shape: np.random.standard_gamma(sh, 9)))
        calls.append((1, 1, None, None, lambda: np.random.standard_normal(1)))
    for a, b in ((1e-5, 1e-5), (2e-15, 5e-15), (0.7, 3.0), (1.0, 1.0), (2.2, 5.5)):
        calls.append((4, 11, a, b, lambda a=a, b=b: np.random.beta(a, b, 11)))
        calls.append((1, 1, None, None, lambda: np.random.standard_normal(1)))
    for kind, n, p1, p2, ref in calls:
        got, want = _draw(nprng, st, kind, n, p1, p2), ref()
        assert np.array_equal(got.view(np.uint64), np.asarray(want, np.float64).view(np.uint64)), (kind, p1, p2, got, want)
        assert np.array_equal(st, numpy_state()), (kind, p1, p2)


@pytest.mark.parametrize("name", _cases()[1])
def test_oracle_perturbed_controls_match_host(built, nprng, name):
    """for each golden case's planned controls and several seeds: the restatement's noisy controls == V.perturbed_controls bit for bit
    (reference order and association) and the streams end in the same state"""
    from mpcmmd_b200 import validation as V
    g, _ = _cases()
    variant, c, num_obs, noise_level, num_prime, noise, key, xt, yt = _case_inputs(g, name)
    prob = _fake_prob(variant, g[name + "_args"])
    acc, steer = V.compute_controls(prob, g[name + "_cx"], g[name + "_cy"])
    for k in (key, 0, 1234567, UINT32_MAX):
        a, s = V.perturbed_controls(prob, acc[:num_prime], steer[:num_prime], noise_level, num_prime, noise, k)
        want_state = numpy_state()
        a_o, s_o, st = oracle_perturbed(nprng, prob, acc[:num_prime], steer[:num_prime], noise_level, num_prime, noise, k)
        assert np.array_equal(a, a_o) and np.array_equal(s, s_o), (name, k)
        assert np.array_equal(st, want_state), (name, k)


def test_device_rng_refuses_nonpositive_beta_shape(built, monkeypatch):
    """beta noise with num_prime = 100 reaches acc[99] == 0, so np.random.beta(2|acc|, ...) raises ValueError("a <= 0"); the device path
    raises the same error from the Python layer, before any library call"""
    from mpcmmd_b200 import binding as B, validation as V
    g, _ = _cases()
    name = "S_beta_solve0"
    args = g[name + "_args"].copy()
    prob = _fake_prob("static", args)
    item = _items(g, [name])
    with pytest.raises(ValueError, match="^a <= 0$"):
        V.compute_stats_batch(prob, item, 100, 0.3, "beta", int(args[1]))                        # the host path: NumPy's own check

    def no_library():
        raise AssertionError("the library must not be called")
    monkeypatch.setattr(B, "load", no_library)
    with pytest.raises(ValueError, match="^a <= 0$"):
        V.compute_stats_batch(prob, item, 100, 0.3, "beta", int(args[1]), rng="device")
    with pytest.raises(ValueError, match="rng='host'"):
        V.compute_stats_batch(prob, item, 50, 0.3, "beta", int(args[1]), rng="device", want_rollouts=True)
    with pytest.raises(ValueError):
        V.compute_stats_batch(prob, item, 50, 0.3, "beta", int(args[1]), rng="gpu")
    bad = [dict(item[0], key=2 ** 32)]
    with pytest.raises(ValueError, match="Seed must be between"):
        V.compute_stats_batch(prob, bad, 50, 0.3, "beta", int(args[1]), rng="device")


def test_parser_rng_flag(built):
    from mpcmmd_b200 import validation as V
    common = ["--noises", "beta", "--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "4", "--num_prime", "50",
              "--acc_const_noise", "0.0", "--steer_const_noise", "0.0"]
    assert V.build_parser().parse_args(common).rng == "host"
    assert V.build_parser().parse_args(common + ["--rng", "device"]).rng == "device"
    with pytest.raises(SystemExit):
        V.build_parser().parse_args(common + ["--rng", "gpu"])


# ---- GPU -------------------------------------------------------------------------------------------------------------------------
def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _host_draws(V, prob, items, num_prime, noise_level, noise):
    """V.perturbed_controls of every item (the host path's draws) and np.random.get_state() after each"""
    acc_p, steer_p, _, _, _, _ = V._inputs(prob, items, num_prime, prob.num_obs)
    a = np.empty((len(items), 1000, num_prime)); s = np.empty_like(a); st = np.empty((len(items), WORDS), np.uint32)
    for i, it in enumerate(items):
        a[i], s[i] = V.perturbed_controls(prob, acc_p[i], steer_p[i], noise_level, num_prime, noise, it["key"])
        st[i] = numpy_state()
    return a, s, st


def _host_counts(V, B, prob, items, num_prime, acc, steer):
    """the host path's counts (compute_stats_batch(rng="host")) from draws already made"""
    _, _, state0, xo, yo, static = V._inputs(prob, items, num_prime, prob.num_obs)
    n = len(items)
    count, lane = np.zeros(n, np.int32), np.zeros(n, np.int32)
    B.check(B.load().mpcmmd_validate_host(prob.device.index or 0, n, 1000, num_prime, prob.num_obs, 1 if static else 0, *V._geometry(prob),
                                          _p(acc), _p(steer), _p(state0), _p(xo), _p(yo), _p(count), _p(lane), None, None))
    return count, lane


def _compare(V, prob, items, num_prime, noise_level, noise, tag):
    """device draws vs host draws: every stream consumed as NumPy consumes it, controls within 1e-12; returns the counts of both
    paths and the largest control difference"""
    from mpcmmd_b200 import binding as B
    a_h, s_h, st_h = _host_draws(V, prob, items, num_prime, noise_level, noise)
    count, lane, a_d, s_d, st_d = V.seeded_stats_batch(prob, items, num_prime, noise_level, noise, prob.num_obs, want_draws=True)
    # consumption (key, pos, has_gauss) exact; the cached, not yet consumed gauss f * x1 carries log's rounding: within 1 ulp
    bad = [i for i in range(len(items)) if not np.array_equal(st_d[i, :626], st_h[i, :626])]
    assert not bad, (tag, "stream consumption differs from NumPy's", bad[:10])
    g_d, g_h = st_d[:, 626:].copy().view(np.float64)[:, 0], st_h[:, 626:].copy().view(np.float64)[:, 0]
    assert np.all(np.abs(g_d - g_h) <= np.spacing(np.abs(g_h))), tag
    err = max(float(np.max(np.abs(a_d - a_h))), float(np.max(np.abs(s_d - s_h))))
    assert err <= 1e-12, (tag, err)
    print("%s: %d streams consumed identically (%d cached gauss 1 ulp apart), max |perturbed control - host| = %.3g"
          % (tag, len(items), int(np.sum(g_d != g_h)), err))
    return (count, lane), _host_counts(V, B, prob, items, num_prime, a_h, s_h), err


@pytest.mark.gpu
@pytest.mark.parametrize("group", ["S_beta", "S_gauss", "D_gauss", "D_beta"])
def test_device_rng_matches_host_on_golden_cases(built, group):
    """all 12 golden cases: every device stream ends in the np.random.get_state() of the host draws; perturbed controls within
    1e-12 absolute of the host's (measured on a B200: at most 4.4e-16, i.e. 1-2 ulp of the controls, where CUDA's pow / log / exp
    round differently from glibc's); counts identical to the reference's (validation_ref.npz)"""
    _need_gpu()
    from mpcmmd_b200 import CEM, binding as B, validation as V
    g, names = _cases()
    names = [n for n in names if n.startswith(group)]
    args = g[names[0] + "_args"]
    variant = "static" if group.startswith("S_") else "dynamic"
    num_obs, noise_level, num_prime, noise = int(args[1]), float(args[2]), int(args[3]), ("gaussian", "beta")[int(args[4])]
    prob = CEM(int(args[0]), num_obs, noise_level, num_prime, noise, float(args[5]), float(args[6]), variant=variant)
    items = _items(g, names)
    (count, lane), (hc, hl), _ = _compare(V, prob, items, num_prime, noise_level, noise, group)
    for i, name in enumerate(names):
        assert [int(count[i]), int(lane[i])] == g[name + "_count"].tolist(), name
    assert np.array_equal(count, hc) and np.array_equal(lane, hl)
    if noise == "beta":                                                  # the library makes np.random.beta's check too
        n = len(items)
        z = np.zeros((n, num_prime)); s0 = np.zeros((n, 5)); o = np.zeros((n, num_obs, num_prime)); cnt = np.zeros(n, np.int32)
        rc = B.load().mpcmmd_validate_seeded_host(0, n, 10, num_prime, num_obs, 1, 1, 0.3, 0.01, 2.0, 5.0, 0.0, 0.0, 0.15, 2.5, 4.25, 2.75,
                                                  -2.25, 2.25, _p(np.zeros(n, np.uint32)), _p(z), _p(z), _p(s0), _p(o), _p(o), _p(cnt),
                                                  _p(cnt.copy()), None, None, None)
        assert rc != 0 and b"a <= 0" in B.load().mpcmmd_last_error()


@pytest.mark.gpu
@pytest.mark.parametrize("variant", ["static", "dynamic"])
def test_device_rng_matches_host_on_solver_plans(built, variant):
    """256 solver-produced plans (128 episodes x {cvar, mmd_opt}; static at configs[1]: O = 4, np = 50, dynamic at configs[2]: O = 6,
    np = 60), seeds 0..255, both noise kinds: not one stream may consume differently from NumPy (a mismatch would mean a libm
    difference flipped a rejection); perturbed controls within 1e-12 absolute (measured on a B200: at most 9.4e-15, dynamic beta
    steering in Johnk's log-space branch, which scales log's error by |log U| / a; 4.4e-16 in the other three runs.  Before
    dnp::pow_np, CUDA's pow in the subnormal range moved single steering draws by up to 0.015 here); counts identical to the host path"""
    _need_gpu()
    from mpcmmd_b200 import CEM, scenes, validation as V
    num_obs, num_prime = (4, 50) if variant == "static" else (6, 60)
    prob = CEM(5, num_obs, 0.3, num_prime, "beta", 0.0, 0.0, variant=variant, max_episodes=128)
    eps = list(range(128))
    batch = scenes.static_batch(prob, eps, variant)
    init_state = scenes.driver_inputs(variant)[0].astype(np.float64)
    items = []
    for cost in ("cvar", "mmd_opt"):
        out = prob.solve_batch(cost, **batch)
        for k in eps:
            it = dict(cx=out["cx"][k].astype(np.float64), cy=out["cy"][k].astype(np.float64), init_state=init_state, key=len(items))
            if variant == "static":
                (x, y, vx, vy, _), _ = scenes.static_scene(num_obs, k)
                it.update(x_obs=x, y_obs=y, vx_obs=vx, vy_obs=vy)
            else:
                _, _, xt, yt = scenes.dynamic_scene(num_obs, k)
                it.update(x_obs_traj=xt.astype(np.float64), y_obs_traj=yt.astype(np.float64))
            items.append(it)
    for noise, noise_level in (("beta", 0.3), ("gaussian", 0.1)):
        (count, lane), (hc, hl), _ = _compare(V, prob, items, num_prime, noise_level, noise, "%s %s" % (variant, noise))
        assert np.array_equal(count, hc) and np.array_equal(lane, hl), (variant, noise)


@pytest.mark.gpu
def test_run_validation_device_rng_matches_host(built, tmp_path):
    """the README workflow (5 static episodes, cvar + mmd_opt) validated with --rng device writes the same stats file as --rng host"""
    _need_gpu()
    from mpcmmd_b200 import driver, validation as V
    common = ["--noises", "beta", "--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "4", "--num_prime", "50",
              "--acc_const_noise", "0.0", "--steer_const_noise", "0.0", "--root", str(tmp_path / "data")]
    driver.run_sweep(driver.build_parser().parse_args(common + ["--costs", "cvar", "mmd_opt", "--num_configs", "5"]), log=lambda *a: None)
    files = {}
    for rng in ("host", "device"):
        args = V.build_parser().parse_args(common + ["--stats_root", str(tmp_path / rng), "--rng", rng])
        files[rng], = V.run_validation(args, "static", log=lambda *a: None)
    h, d = np.load(files["host"]), np.load(files["device"])
    assert set(h.files) == set(d.files) and len(h["coll_cvar"]) >= 1
    for k in h.files:
        assert np.array_equal(h[k], d[k]), k
