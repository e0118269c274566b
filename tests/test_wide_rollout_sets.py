"""cvar, saa and mmd_random with 65..1024 rollouts per CEM sample (k_rollouts_wide, one CTA per sample) against the CPU reference of
tests/wide_oracle/oracle_wide.c, bit for bit.

Sizes: the warp edges 65, 96 / 97, 128 / 129 and 1023 / 1024; 101 and 1001, where q = 0.98 (nr - 1) is an integer in float32 (lo == hi);
the others interpolate.  Scenes: an obstacle on the path, no collision at all (var = 0: every rollout is in the CVaR tail) and every rollout
colliding.  NaN rollouts at chosen indices come in through injected Beta draws.  Launch sizes 1, 100 and more than 2 x SMs samples must give
the same bits.  Full solves (also grouped and batched episodes), the refusals, a 200-episode create and the sweep driver complete the
picture."""
import os

import numpy as np
import pytest

import wide_ref as W

pytestmark = pytest.mark.gpu
f32 = np.float32
ST0 = np.array([0.0, 1.75, 5.0, 0.0, 0.0], f32)
SMALL = dict(num_batch=24, maxiter_cem=3)
SIZES = [65, 96, 97, 101, 128, 129, 255, 256, 511, 1001, 1023, 1024]


def _eq(a, b, what=""):
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if not np.array_equal(a, b, equal_nan=True):
        bad = np.flatnonzero(~((a == b) | (np.isnan(a) & np.isnan(b))).ravel())
        raise AssertionError(f"{what}: {bad.size}/{a.size} elements differ; first at {bad[:5]}: got {a.ravel()[bad[:5]]} want {b.ravel()[bad[:5]]}")


@pytest.fixture(scope="module")
def mods(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mpcmmd_b200 import cem_impl
    from oracle import oracle as O
    O.set_threads(min(32, os.cpu_count() or 1))
    return cem_impl, O


@pytest.fixture(scope="module")
def wl(mods, tmp_path_factory):
    return W.build_lib(tmp_path_factory.mktemp("wide_oracle"))


@pytest.fixture(scope="module")
def sms(mods):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _pair(mods, wl, nr, args, max_episodes=1, kernel="laplace", **kw):
    cem_impl, O = mods
    return cem_impl.CEM(nr, *args, max_episodes=max_episodes, kernel=kernel, **kw), W.WideOracle(O, wl, nr, *args, kernel=kernel, **kw)


def _controls(ora, rng, n, bases=12):
    beq_x = np.array([0.0, 5.0, 0.0], f32); beq_y = np.array([1.75, 0.0, 0.0, 0.0], f32)
    acc, steer = [], []
    for _ in range(min(n, bases)):
        p = np.concatenate([rng.uniform(2, 25, 4), rng.normal(0, 3, 4)]).astype(f32)
        o = ora.project(p, beq_x, beq_y, 15.0, np.zeros(11, f32), np.zeros(11, f32), np.zeros(198, f32))
        acc.append(o["acc"]); steer.append(o["steer"])
    acc, steer = np.stack(acc), np.stack(steer)
    if n <= bases:
        return acc, steer
    pick = rng.integers(0, bases, n)
    return ((acc[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32), (steer[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32))


def _scene(O, ora, kind="path"):
    xo, yo, _ = ora.compute_obs_trajectories(*O.static_scene(2, 5))
    xo = xo.copy(); yo = yo.copy()
    if kind == "path":                     # an obstacle on the path: some rollouts collide
        xo[0] = np.linspace(2, 60, 100); yo[0] = 1.75
    elif kind == "clear":                  # nothing within reach: every cost is 0, var = 0
        xo[:] = 1.0e3
    else:                                  # "all": an obstacle 1 m beside the start point, so every rollout's first knot already has cost 0.87
        xo[0] = np.linspace(0, 60, 100); yo[0] = 2.75
    return np.ascontiguousarray(xo, f32), np.ascontiguousarray(yo, f32)


def _oracle(wide, cost, acc, steer, noise_t, xo, yo, idx, draws=None):
    from concurrent.futures import ThreadPoolExecutor
    idx = [int(i) for i in idx]
    def one(i):
        bd = None if draws is None else (draws[0][i], draws[1][i])
        return wide.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo, beta_draws=bd)
    with ThreadPoolExecutor(max_workers=max(1, min(len(idx), os.cpu_count() or 1))) as ex:
        return dict(zip(idx, ex.map(one, idx)))


def _fields(cost):
    return ("risk", "lane", "beta", "sigma") if cost == "mmd_random" else ("risk", "lane")


def _check(got, refs, cost, what):
    for i, ref in refs.items():
        for k in _fields(cost):
            _eq(got[k][i], ref[k], f"{what} sample {i} {k}")


def _parts(prob, cost, acc, steer, noise_t, xo, yo, size):
    outs = [prob.stage_risk(cost, acc[a:a + size], steer[a:a + size], ST0, noise_t, xo, yo) for a in range(0, len(acc), size)]
    return {k: np.concatenate([o[k] for o in outs]) for k in outs[0]}


# ---------------------------------------------------------------------------------------------------------------------------------
# stage risk

CASES = ([(c, nr, "gaussian", "laplace") for c in ("cvar", "saa", "mmd_random") for nr in SIZES]
         + [(c, nr, "beta", "laplace") for c in ("cvar", "saa", "mmd_random") for nr in (65, 97, 101, 256, 1001, 1024)]
         + [("mmd_random", nr, "gaussian", "gaussian") for nr in (129, 1024)])


@pytest.mark.parametrize("cost,nr,noise,kernel", CASES)
def test_stage_risk_wide(mods, wl, sms, cost, nr, noise, kernel):
    """one launch of 2 x SMs + 5 samples equals launches of 100 samples and of single samples, and sampled samples equal the CPU reference
    (kernel: the MMD kernel form, which only mmd_random reads)"""
    cem_impl, O = mods
    n = 2 * sms + 5
    prob, wide = _pair(mods, wl, nr, (2, 0.3 if noise == "beta" else 0.1, 20, noise, 0.05, 0.01), max_episodes=-(-n // 100), kernel=kernel)
    acc, steer = _controls(wide, np.random.default_rng(7000 + nr), n)
    noise_t = wide.noise_tables(91, 2)
    xo, yo = _scene(O, wide)
    got = prob.stage_risk(cost, acc, steer, ST0, noise_t, xo, yo)
    for k in _fields(cost):
        assert got[k].shape[0] == n
    by100 = _parts(prob, cost, acc, steer, noise_t, xo, yo, 100)
    for k in _fields(cost):
        _eq(got[k], by100[k], f"{cost} nr={nr} {k}: one launch of {n} vs launches of 100")
    single = [2, n - 1]
    for i in single:
        one = prob.stage_risk(cost, acc[i:i + 1], steer[i:i + 1], ST0, noise_t, xo, yo)
        for k in _fields(cost):
            _eq(got[k][i], one[k][0], f"{cost} nr={nr} {k}: sample {i} alone")
    pick = sorted({0, 1, 2, n // 2, n - 1} | {int(i) for i in np.linspace(3, n - 2, 5 if nr > 256 else 11)})
    _check(got, _oracle(wide, cost, acc, steer, noise_t, xo, yo, pick), cost, f"{cost} nr={nr} {noise} {kernel}")
    assert np.isfinite(got["risk"]).all()
    if cost == "cvar":
        assert np.any(got["risk"] != got["risk"][0])


@pytest.mark.parametrize("scene", ["clear", "all"])
@pytest.mark.parametrize("nr", [65, 101, 1024])
@pytest.mark.parametrize("cost", ["cvar", "saa", "mmd_random"])
def test_stage_risk_wide_scenes(mods, wl, cost, nr, scene):
    """no collision (every cost 0: var = 0, the whole set is the CVaR tail and every tail term is a skipped zero) and every rollout colliding"""
    cem_impl, O = mods
    prob, wide = _pair(mods, wl, nr, (2, 0.1, 20, "gaussian", 0.05, 0.01), max_episodes=1)
    acc, steer = _controls(wide, np.random.default_rng(8000 + nr), 7)
    noise_t = wide.noise_tables(17, 1)
    xo, yo = _scene(O, wide, scene)
    got = prob.stage_risk(cost, acc, steer, ST0, noise_t, xo, yo)
    refs = _oracle(wide, cost, acc, steer, noise_t, xo, yo, range(7))
    _check(got, refs, cost, f"{cost} nr={nr} scene {scene}")
    costs = np.stack([refs[i]["red_cost"] for i in range(7)])
    if scene == "clear":
        assert (costs == 0).all()
    else:
        assert (costs > 0).all()


@pytest.mark.parametrize("nr", [65, 97, 129, 256, 1024])
@pytest.mark.parametrize("cost", ["cvar", "saa", "mmd_random"])
def test_stage_risk_wide_nan_rollouts(mods, wl, cost, nr):
    """NaN Beta draws at chosen (sample, rollout) pairs, warp boundaries included, through mpcmmd_stage_risk_injected: the rollout's costs are
    NaN, which sorts last in the CVaR order statistics, does not count in saa and propagates through the MMD"""
    cem_impl, O = mods
    np_ = 20
    prob, wide = _pair(mods, wl, nr, (2, 0.3, np_, "beta", 0.05, 0.01), max_episodes=1)
    rng = np.random.default_rng(9000 + nr)
    n = 6
    acc, steer = _controls(wide, rng, n)
    z3 = wide.noise_tables(5, 0)[2]
    b1 = rng.beta(2.0, 5.0, (n, nr * np_)).astype(f32); b2 = rng.beta(2.0, 5.0, (n, nr * np_)).astype(f32)
    rows = [r for r in (0, 31, 32, 63, 64, 95, 96, 127, 128, nr - 2, nr - 1) if r < nr]
    for s in range(1, n):                           # sample 0 keeps finite draws; sample s gets the first s of the chosen rows
        for r in rows[:2 * s]:
            b1[s, r * np_ + (r % np_)] = np.nan
    b2[n - 1, :np_] = np.nan                        # and the last sample also a NaN steering row
    xo, yo = _scene(O, wide)
    got = prob.stage_risk_injected(cost, acc, steer, ST0, z3, b1, b2, xo, yo)
    noise_t = (z3, z3, z3, None, [0, 0, 0, 0])
    refs = _oracle(wide, cost, acc, steer, noise_t, xo, yo, range(n), draws=(b1, b2))
    _check(got, refs, cost, f"{cost} nr={nr} NaN rollouts")
    assert np.isnan(refs[n - 1]["red_cost"]).sum() >= 2


def test_stage_noise_wide(mods, wl):
    """the per-iteration noise tables of a num_reduced > 64 handle (k_noise_wide) equal the oracle's"""
    cem_impl, O = mods
    prob, wide = _pair(mods, wl, 300, (2, 0.3, 50, "beta", 0.05, 0.01), max_episodes=2)
    for idx, it in ((4242, 0), (17, 7), (1, 19)):
        got = prob.stage_noise(idx, it); ref = wide.noise_tables(idx, it)
        for a, b, k in zip(got, ref, ("z1", "z2", "z3", "z_cem", "keys")):
            _eq(np.asarray(a), np.asarray(b), f"idx {idx} it {it} {k}")


# ---------------------------------------------------------------------------------------------------------------------------------
# full solves

def _inputs(O, wide, E, num_obs=2):
    eps = [O.static_episode(num_obs, k) for k in range(E)]
    tr = [wide.compute_obs_trajectories(*sc) for sc, _ in eps]
    init_state, mean, cov, v_des = O.driver_inputs("static")
    return dict(idx_mpc=[i for _, i in eps], init_state=np.stack([init_state] * E), mean_param=np.stack([mean] * E),
                cov_param=np.stack([cov] * E), x_obs_traj=np.stack([t[0] for t in tr]), y_obs_traj=np.stack([t[1] for t in tr]),
                v_des=[v_des] * E)


def _ref_solve(wide, cost, b, e):
    return wide.solve(cost, b["idx_mpc"][e], b["init_state"][e], b["mean_param"][e], b["cov_param"][e], b["x_obs_traj"][e], b["y_obs_traj"][e],
                      b["v_des"][e])


SOLVE_KEYS = ("cx", "cy", "cost_obs", "cost_lane")


@pytest.mark.parametrize("cost,nr,noise", [(c, nr, nz) for c in ("cvar", "saa") for nr in (128, 1024) for nz in ("gaussian", "beta")]
                         + [("mmd_random", 128, nz) for nz in ("gaussian", "beta")] + [("mmd_random", 1024, "gaussian")])
def test_solve_wide(mods, wl, cost, nr, noise):
    cem_impl, O = mods
    E = 3
    prob, wide = _pair(mods, wl, nr, (2, 0.3 if noise == "beta" else 0.1, 30, noise, 0.02, 0.01), max_episodes=E, **SMALL)
    b = _inputs(O, wide, E)
    got = prob.solve_batch(cost, **b)
    for e in range(E):
        ref = _ref_solve(wide, cost, b, e)
        for k in SOLVE_KEYS + (("beta", "sigma") if cost == "mmd_random" else ()):
            _eq(got[k][e], ref[k], f"{cost} nr={nr} {noise} ep{e} {k}")
    assert np.isfinite(got["cx"]).all()


def test_solve_wide_reference_sizes(mods, wl):
    """cvar at num_reduced 256 with the reference's 100 samples x 20 iterations"""
    cem_impl, O = mods
    prob, wide = _pair(mods, wl, 256, (4, 0.3, 50, "beta", 0.0, 0.0), max_episodes=1)
    b = _inputs(O, wide, 1, num_obs=4)
    got = prob.solve_batch("cvar", **b)
    ref = _ref_solve(wide, "cvar", b, 0)
    for k in SOLVE_KEYS:
        _eq(got[k][0], ref[k], f"cvar nr=256 100 x 20 {k}")


def test_solve_wide_batched_and_grouped_episodes_equal_alone(mods, wl, monkeypatch):
    """5 episodes in one solve, and in a graph split into 3 episode groups (MPCMMD_GROUPS=3: every group views its own episodes' single noise
    slot), equal each episode solved alone and the CPU reference"""
    cem_impl, O = mods
    E = 5
    args = (2, 0.3, 30, "beta", 0.02, 0.01)
    prob, wide = _pair(mods, wl, 128, args, max_episodes=E, **SMALL)
    monkeypatch.setenv("MPCMMD_GROUPS", "3")
    grouped = cem_impl.CEM(128, *args, max_episodes=E, **SMALL)
    monkeypatch.delenv("MPCMMD_GROUPS")
    one = cem_impl.CEM(128, *args, max_episodes=1, **SMALL)
    b = _inputs(O, wide, E)
    out = prob.solve_batch("cvar", **b)
    outg = grouped.solve_batch("cvar", **b)
    assert grouped.last_launch_count() > prob.last_launch_count()        # the grouped graph has three copies of the setup kernels
    for e in range(E):
        solo = one.solve_batch("cvar", **{k: v[e:e + 1] for k, v in b.items()})
        ref = _ref_solve(wide, "cvar", b, e)
        for k in SOLVE_KEYS:
            _eq(out[k][e], solo[k][0], f"episode {e} {k}: batched vs alone")
            _eq(outg[k][e], solo[k][0], f"episode {e} {k}: grouped vs alone")
            _eq(out[k][e], ref[k], f"episode {e} {k}: vs CPU reference")


# ---------------------------------------------------------------------------------------------------------------------------------
# creation and refusals

def test_wide_refusals(mods):
    cem_impl, O = mods
    from mpcmmd_b200 import binding as B
    from mpcmmd_b200 import scenes
    with pytest.raises(B.MpcmmdError, match=r"num_reduced must be in \[2,1024\]"):
        cem_impl.CEM(1025, 2, 0.1, 20, "gaussian", 0.0, 0.0, max_episodes=1, num_batch=24)
    for nr in (41, 65, 1024):                        # mmd_opt stays at num_reduced <= 40
        p = cem_impl.CEM(nr, 2, 0.1, 20, "gaussian", 0.0, 0.0, max_episodes=1, num_batch=24, maxiter_cem=1)
        with pytest.raises(B.MpcmmdError, match=r"mmd_opt: num_reduced must be in \[2, 40\]"):
            p.solve_batch("mmd_opt", **scenes.static_batch(p, [0]))
        if nr > 64:
            with pytest.raises(B.MpcmmdError, match="no inner-CEM tables"):
                p.tables()
        del p


def test_wide_create_200_episodes_fits(mods):
    """200 episodes at num_reduced 1024, num_prime 100, beta noise: the noise tables hold one outer iteration per episode (about 3.9 GB), so
    the handle creates"""
    cem_impl, O = mods
    p = cem_impl.CEM(1024, 4, 0.3, 100, "beta", 0.0, 0.0, max_episodes=200)
    assert p.num_reduced == 1024 and p.max_episodes == 200
    del p


# ---------------------------------------------------------------------------------------------------------------------------------
# the sweep driver

def test_sweep_driver_wide(mods, wl, tmp_path):
    """main_mpc.py's loop at --num_reduced_sets 128 for cvar, saa and mmd_random: the reference's file names and keys, and the accepted
    episodes' plans equal the CPU reference's solves"""
    cem_impl, O = mods
    from mpcmmd_b200 import driver
    argv = ["--costs", "cvar", "saa", "mmd_random", "--noises", "beta", "--noise_levels", "0.3", "--num_reduced_sets", "128", "--num_obs", "2",
            "--num_prime", "30", "--acc_const_noise", "0.0", "--steer_const_noise", "0.0", "--num_configs", "3", "--root", str(tmp_path)]
    written = driver.run_sweep(driver.build_parser().parse_args(argv), log=lambda *a: None)
    assert written == [str(tmp_path / "beta_noise" / "noise_30" / "ts_30" / f"{c}_128_samples_2_obs.npz") for c in ("cvar", "saa", "mmd_random")]
    wide = W.WideOracle(O, wl, 128, 2, 0.3, 30, "beta", 0.0, 0.0)
    init_state, mean, cov, v_des = O.driver_inputs("static")
    refs = {}
    for cost, path in zip(("cvar", "saa", "mmd_random"), written):
        data = np.load(path)
        assert set(data.files) == {"cx", "cy", "init_state", "x_obs", "y_obs", "vx_obs", "vy_obs"}
        solver = "mmd_random" if cost == "mmd_random" else "cvar"          # main_mpc.py runs compute_cem_cvar for saa
        thr = -1000.0 + 1.0 if cost == "mmd_random" else 1e-5
        rows = []
        for k in range(3):
            sc, idx = O.static_episode(2, k)
            xt, yt, _ = wide.compute_obs_trajectories(*sc)
            key = (solver, k)
            if key not in refs:
                refs[key] = wide.solve(solver, idx, init_state, mean, cov, xt, yt, v_des)
            if refs[key]["cost_obs"] <= thr:
                rows.append(refs[key])
        assert data["cx"].shape == (len(rows), 11)
        for r, ref in enumerate(rows):
            _eq(data["cx"][r].astype(f32), ref["cx"], f"{cost} row {r} cx"); _eq(data["cy"][r].astype(f32), ref["cy"], f"{cost} row {r} cy")
