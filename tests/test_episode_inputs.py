"""Batched solves whose episodes differ in every per-episode input, each episode against its own oracle solve.

mpcmmd_solve takes seven inputs per episode: idx_mpc, init_state (E, 6), mean_param (E, 8), cov_param (E, 8, 8), the obstacle trajectories
and v_des (E,).  Every kernel of the solve reads its episode's slice of them: k_boundary (init_state -> beq_x, beq_y, state0 with the heading
atan2(vy, vx)), k_init (mean0, cov0), k_project / k_project_tc (beq_x + 3 e, beq_y + 4 e, v_des[e]), the rollout bodies, k_opt_risk,
k_rollouts_wide and the inner-CEM kernels (state0 + 5 e), k_select (mean + 8 e, cov + 64 e), and push_view offsets all of them for the
episode groups of a grouped solve graph.  A solve whose episodes share those inputs cannot tell a read of episode e from a read of episode
0, so the batches here give every episode its own initial state, CEM mean and covariance, v_des, scene and idx_mpc (`episode_inputs`).

A CPU test shows, on the oracle alone, that each of these fields moves the solve at the sizes used here, so a kernel that reads another
episode's field cannot match the oracle by chance.  The GPU cells compare every episode (or the marked ones of the large launches) with the
oracle bit for bit, and assert by name the rollout / inner-CEM instantiation a launch-size-dependent cell reaches.  At full size the
checks are oracle-free: a permuted batch gives permuted outputs bit for bit, and each plan meets its own boundary conditions (also under the
tensor-core projection, whose trajectories are not bit-comparable).  Handle reuse, the CUDA-tensor entry point on torch streams and the
Monte-Carlo validation with per-plan initial states close the module.

Not covered: k_inner_cem_big with more chains than one chunk of its scratch (num_reduced >= 30), where the oracle is too slow."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import kernel_names as KN
import wide_ref as W

gpu = pytest.mark.gpu
f32 = np.float32
ROLL_THREADS = 128                                                     # k_rollouts CTA size (csrc/k_risk.cuh)
SMALL = dict(num_batch=24, maxiter_cem=3, num_samples_cem=40, maxiter_beta_cem=4)
GROUPED = dict(num_batch=100, maxiter_cem=2, num_samples_cem=40, maxiter_beta_cem=4)
FULL_ARGS = (5, 4, 0.3, 50, "beta", 0.0, 0.0)                         # BASELINE configs[1]
FIELDS = ("x0", "y0", "vx", "vy", "ax", "ay", "mean", "cov", "v_des")
BC_TOL = 2e-3                                                          # the boundary-condition tolerance of test_projection_properties


def _keys(cost):
    return ("cx", "cy", "cost_obs", "cost_lane") + (("beta", "sigma", "res_beta") if cost == "mmd_opt" else ())


def _args(nr=5, nobs=2, noise="gaussian", np_=30):
    return (nr, nobs, 0.3 if noise == "beta" else 0.1, np_, noise, 0.02, 0.01)


# ---------------------------------------------------------------------------------------------------------------------------------
# input generator

def _strata(rng, E, lo, hi):
    """E values in [lo, hi], one per stratum of width (hi - lo) / E in random order, each within the middle fifth of its stratum: any two
    differ by at least 0.8 (hi - lo) / E"""
    return lo + (rng.permutation(E) + rng.uniform(0.4, 0.6, E)) * (hi - lo) / E


def _signed(rng, E, lo, hi):
    """stratified magnitudes in [lo, hi] with random signs: never 0, any two at least 0.8 (hi - lo) / E apart"""
    return _strata(rng, E, lo, hi) * rng.choice([-1.0, 1.0], E)


def _scene(ora, k, variant):
    """(idx_mpc, x_obs_traj, y_obs_traj) of scene k: the reference's generators for up to 9 obstacles, the scaled one above"""
    from mpcmmd_b200 import scenes
    if variant == "dynamic":
        _, idx, xt, yt = scenes.dynamic_scene(ora.num_obs, k)
        return idx, xt, yt
    sc, idx = scenes.static_scene(ora.num_obs, k) if ora.num_obs <= 9 else scenes.scaled_scene(ora.num_obs, k)
    xt, yt, _ = ora.compute_obs_trajectories(*sc)
    return idx, xt, yt


def episode_inputs(ora, E, seed, variant="static"):
    """solve_batch inputs of E episodes, every per-episode field its own.  Episode 0 carries the driver's defaults (main_mpc.py), episode 1
    an initial heading outside (-pi/2, pi/2), episodes 2 and 3 the same scene and idx_mpc with different state, mean, covariance and v_des;
    the others: x0 in [-4, 4], y0 within 0.45 of the lane (static: either lane, dynamic: lane -1.75, inside y_ub = -1.25), vx in [2, 10],
    vy, ax, ay nonzero of either sign, mean speeds in [8, 22] with nonzero lateral entries, an SPD covariance with its own diagonal and
    nonzero correlations (exactly symmetric in float32), v_des in [8, 22]"""
    from oracle import oracle as O
    rng = np.random.default_rng(seed)
    lane = -1.75 if variant == "dynamic" else rng.choice([-1.75, 1.75], E)
    h = 0.45 / E                                                       # half a y0 stratum: the lane centre is the middle of one
    st = np.stack([_strata(rng, E, -4.0, 4.0), lane + _strata(rng, E, -0.45 - h, 0.45 - h), _strata(rng, E, 2.0, 10.0),
                   _signed(rng, E, 0.1, 1.2), _signed(rng, E, 0.1, 2.0), _signed(rng, E, 0.1, 1.5)], 1)
    d_st, d_mean, d_cov, d_vdes = O.driver_inputs(variant)
    for j in range(6):                          # the episode whose value is nearest the default's takes episode 0's: the default gets a stratum of its own
        i = 1 + int(np.argmin(np.abs(st[1:, j] - d_st[j])))
        st[i, j] = st[0, j]
    mean = np.concatenate([rng.uniform(8.0, 22.0, (E, 4)), _signed(rng, 4 * E, 0.2, 1.5).reshape(E, 4)], 1)
    cov = np.empty((E, 8, 8))
    for e in range(E):
        d = np.sqrt(np.concatenate([rng.uniform(10.0, 30.0, 4), rng.uniform(50.0, 150.0, 4)]))
        r = rng.uniform(-0.12, 0.12, (8, 8))
        r = (r + r.T) / 2
        np.fill_diagonal(r, 1.0)                                       # off-diagonal row sums < 1: diagonally dominant, so SPD
        cov[e] = d[:, None] * r * d[None]
    v_des = _strata(rng, E, 8.0, 22.0)
    scene_of = list(range(E))
    st[1, 2] = -st[1, 2]                                               # vx < 0: heading in (pi/2, pi] or [-pi, -pi/2)
    if E > 3:
        scene_of[3] = scene_of[2]
    st[0], mean[0], cov[0], v_des[0] = d_st, d_mean, d_cov, d_vdes
    cov = cov.astype(f32)
    cov = np.triu(cov) + np.swapaxes(np.triu(cov, 1), 1, 2)
    scenes_ = [_scene(ora, 1000 * seed + k, variant) for k in scene_of]
    return dict(idx_mpc=np.array([s[0] for s in scenes_], np.int32), init_state=st.astype(f32), mean_param=mean.astype(f32), cov_param=cov,
                x_obs_traj=np.stack([s[1] for s in scenes_]).astype(f32), y_obs_traj=np.stack([s[2] for s in scenes_]).astype(f32),
                v_des=v_des.astype(f32))


def _sub(b, idx):
    return {k: v[idx] for k, v in b.items()}


def _with_field(b, k, src, field):
    """b with episode k's `field` replaced by episode src's"""
    b = {n: v.copy() for n, v in b.items()}
    if field in FIELDS[:6]:
        b["init_state"][k, FIELDS.index(field)] = b["init_state"][src, FIELDS.index(field)]
    else:
        name = {"mean": "mean_param", "cov": "cov_param", "v_des": "v_des"}[field]
        b[name][k] = b[name][src]
    return b


# ---------------------------------------------------------------------------------------------------------------------------------
# helpers

def _eq(a, b, what=""):
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if not np.array_equal(a, b, equal_nan=True):
        bad = np.flatnonzero(~((a == b) | (np.isnan(a) & np.isnan(b))).ravel())
        raise AssertionError(f"{what}: {bad.size}/{a.size} elements differ; first at {bad[:5]}: got {a.ravel()[bad[:5]]} want {b.ravel()[bad[:5]]}")


def _pool(fn, idx):
    idx = [int(i) for i in idx]
    with ThreadPoolExecutor(max_workers=max(1, min(len(idx), os.cpu_count() or 1))) as ex:
        return dict(zip(idx, ex.map(fn, idx)))


def _ref(ora, cost, b, e):
    return ora.solve(cost, int(b["idx_mpc"][e]), b["init_state"][e], b["mean_param"][e], b["cov_param"][e], b["x_obs_traj"][e],
                     b["y_obs_traj"][e], float(b["v_des"][e]))


def _check(got, ora, cost, b, what, idx=None):
    """episodes idx (all by default) of `got` equal the oracle's solves of their own inputs, bit for bit"""
    E = len(b["idx_mpc"])
    refs = _pool(lambda e: _ref(ora, cost, b, e), range(E) if idx is None else sorted(set(idx)))
    for e, ref in refs.items():
        for k in _keys(cost):
            _eq(got[k][e], ref[k] if k != "res_beta" else ref[k][:got[k].shape[1]], f"{what}: episode {e} {k}")
    return refs


def _same(a, b, cost, what):
    for k in _keys(cost):
        _eq(a[k], b[k], f"{what} {k}")


def _launch(fn, want, what):
    """fn() under the profiler; asserts that every instantiation in `want` ran"""
    out, names = KN.launched(fn)
    ran = KN.family(names, "rollout") | KN.family(names, "inner")
    missing = set(want) - ran
    assert not missing, f"{what}: expected {sorted(want)} to run, the profiler saw {sorted(ran)} (all kernels: {sorted(names)})"
    return out


def _twins_differ(got, cost, what):
    """episodes 2 and 3 share scene and idx_mpc, not state, mean or v_des: their plans differ"""
    assert any(not np.array_equal(got[k][2], got[k][3]) for k in ("cx", "cy")), f"{what}: episodes 2 and 3 gave the same plan"


@pytest.fixture(scope="module")
def ora_mod(built):
    from oracle import oracle as O
    O.set_threads(min(32, os.cpu_count() or 1))
    return O


@pytest.fixture(scope="module")
def mods(ora_mod):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mpcmmd_b200 import cem_impl
    return cem_impl, ora_mod


@pytest.fixture(scope="module")
def sms(mods):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def wl(mods, tmp_path_factory):
    return W.build_lib(tmp_path_factory.mktemp("wide_oracle"))


@pytest.fixture(scope="module")
def gk(mods, tmp_path_factory):
    """tests/gauss_oracle/oracle_gauss.c built with the oracle's flags into a temporary directory"""
    import ctypes as C
    import subprocess
    out = str(tmp_path_factory.mktemp("gauss_oracle") / "liboracle_gauss.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                           "-Wall", "-Wno-unused-function", "-Wno-misleading-indentation", "-Wno-maybe-uninitialized",
                           os.path.join(os.path.dirname(os.path.abspath(__file__)), "gauss_oracle", "oracle_gauss.c"), "-o", out, "-lm"])
    lib = C.CDLL(out)
    lib.oracle_set_threads(min(32, os.cpu_count() or 1))
    return lib


def _handle(mods, monkeypatch, args, E, env=None, **kw):
    """a CEM handle of E episodes; `env` (MPCMMD_INNER_CEM, MPCMMD_GROUPS, MPCMMD_PROJ) is read at create"""
    cem_impl, _ = mods
    for k in ("MPCMMD_INNER_CEM", "MPCMMD_GROUPS", "MPCMMD_PROJ", "MPCMMD_MATH"):
        monkeypatch.delenv(k, raising=False)
    for k, v in (env or {}).items():
        monkeypatch.setenv(k, v)
    prob = cem_impl.CEM(*args, max_episodes=E, **kw)
    for k in (env or {}):
        monkeypatch.delenv(k)
    return prob


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: the generator, and each per-episode field moves the oracle's solve

def test_generator_separates_episodes(built):
    """the 200-episode batch of the full-size checks: every field of every episode its own, each boundary value further than BC_TOL from
    every other episode's, the heading of episode 1 outside (-pi/2, pi/2), episodes 2 and 3 sharing only scene and idx_mpc, each
    covariance symmetric and positive definite in float32"""
    from oracle import oracle as O
    ora = O.OracleCEM(*FULL_ARGS)
    for variant, E, seed in (("static", 200, 7), ("dynamic", 5, 3)):
        b = episode_inputs(ora if variant == "static" else O.OracleCEM(*_args(nobs=2), variant="dynamic"), E, seed, variant)
        st = b["init_state"].astype(np.float64)
        for j in range(6):
            gap = np.diff(np.sort(st[:, j])).min()
            assert gap > 1.5 * BC_TOL, (variant, FIELDS[j], gap)
        assert abs(np.arctan2(st[1, 3], st[1, 2])) > np.pi / 2
        assert np.all(b["cov_param"] == np.swapaxes(b["cov_param"], 1, 2))
        assert np.linalg.eigvalsh(b["cov_param"].astype(np.float64)).min() > 1.0
        assert len(np.unique(b["v_des"])) == E and len(np.unique(b["mean_param"][:, 0])) == E
        assert b["idx_mpc"][2] == b["idx_mpc"][3] and np.array_equal(b["x_obs_traj"][2], b["x_obs_traj"][3])
        if variant == "dynamic":
            assert np.all(st[:, 1] < -1.25) and np.all(st[:, 1] > -2.25)


@pytest.mark.parametrize("cost", ["cvar", "mmd_opt"])
def test_every_field_moves_the_oracle_solve(ora_mod, cost):
    """for each per-episode field, episode 4 of the small-size batch solved with episode 0's value of that field gives another plan or
    cost than with its own: a kernel that read the field at episode 0 could not match the oracle (the GPU cells below use these sizes)"""
    O = ora_mod
    ora = O.OracleCEM(*_args(), **SMALL)
    b = episode_inputs(ora, 5, 1)
    k = 4
    base = _ref(ora, cost, b, k)
    moved = _pool(lambda j: _ref(ora, cost, _with_field(b, k, 0, FIELDS[j]), k), range(len(FIELDS)))
    for j, r in moved.items():
        assert any(not np.array_equal(r[n], base[n], equal_nan=True) for n in _keys(cost)), f"{cost}: {FIELDS[j]} of episode 0 gives the same solve"


# ---------------------------------------------------------------------------------------------------------------------------------
# B1: small sizes, every cost and noise

SMALL_CASES = [(c, n, "static") for c in ("cvar", "saa", "mmd_random", "mmd_opt") for n in ("gaussian", "beta")] + \
              [("cvar", "gaussian", "dynamic"), ("mmd_opt", "beta", "dynamic")]
NZ = {"gaussian": 0, "beta": 1}                                       # NZ of a solve launch: the Beta candidate table with beta noise


@gpu
@pytest.mark.parametrize("cost,noise,variant", SMALL_CASES)
def test_small_sizes(mods, sms, monkeypatch, cost, noise, variant):
    """five episodes at 24 samples: mmd_opt runs the folding latency body and k_inner_cem_lat (120 chains <= SMs), the others
    k_rollouts<ROLL_STAGED>; every episode equals its oracle solve"""
    _, O = mods
    E = 5
    assert E * SMALL["num_batch"] <= sms
    prob = _handle(mods, monkeypatch, _args(noise=noise), E, variant=variant, **SMALL)
    ora = O.OracleCEM(*_args(noise=noise), variant=variant, **SMALL)
    b = episode_inputs(ora, E, 11 + len(cost), variant)
    want = {f"k_rollouts<0, false, {NZ[noise]}, 2>", "k_inner_cem_lat<5, 0, 0, 0>"} if cost == "mmd_opt" else {f"k_rollouts<2, false, {NZ[noise]}, 0>"}
    got = _launch(lambda: prob.solve_batch(cost, **b), want, f"{cost} {noise} {variant}")
    _check(got, ora, cost, b, f"{cost} {noise} {variant}")
    _twins_differ(got, cost, f"{cost} {noise} {variant}")


# ---------------------------------------------------------------------------------------------------------------------------------
# B2: mmd_opt at each automatic inner-CEM shape

def _inner_cells(sms):
    """cell -> (num_reduced, episodes at num_batch 24, MPCMMD_INNER_CEM, instantiations asserted)"""
    lat_E, fast_E, thr_E = 5, sms // 24 + 1, (3 * sms) // 24 + 1
    return {
        "lat": (5, lat_E, None, {"k_inner_cem_lat<5, 0, 0, 0>", "k_rollouts<0, false, 0, 2>"}),
        "fast_latency": (5, fast_E, None, {"k_inner_cem_fast<5, true, false, 0, 0, 0>", "k_rollouts<0, false, 0, 2>", "k_opt_risk<false>"}),
        "fast_throughput": (5, thr_E, None, {"k_inner_cem_fast<5, false, false, 0, 0, 0>", "k_rollouts<0, false, 0, 0>", "k_opt_risk<false>"}),
        "generic": (5, lat_E, "generic", {"k_inner_cem<5, 0, 0, 0>", "k_rollouts<0, false, 0, 1>"}),
        "nr8": (8, lat_E, None, {"k_inner_cem<8, 0, 0, 0>", "k_rollouts<0, false, 0, 1>"}),
        "nr12_1024": (12, lat_E, None, {"k_inner_cem_big<1024, 0>"}),
        "nr12_256": (12, fast_E, None, {"k_inner_cem_big<256, 0>"}),
    }


@gpu
@pytest.mark.parametrize("cell", ["lat", "fast_latency", "fast_throughput", "generic", "nr8", "nr12_1024", "nr12_256"])
def test_inner_cem_shapes(mods, sms, monkeypatch, cell):
    """mmd_opt with per-episode inputs at <= SMs chains (k_inner_cem_lat, folded risk), (SMs, 3 SMs] (latency build of k_inner_cem_fast),
    > 3 SMs (throughput build, then k_opt_risk), MPCMMD_INNER_CEM=generic, num_reduced 8 (generic kernel on stored mother rollouts) and
    num_reduced 12 (k_inner_cem_big, 1024 threads at <= SMs chains, 256 above): every episode equals its oracle solve"""
    _, O = mods
    nr, E, mode, want = _inner_cells(sms)[cell]
    chains = E * SMALL["num_batch"]
    assert {"lat": chains <= sms, "fast_latency": sms < chains <= 3 * sms, "fast_throughput": chains > 3 * sms,
            "nr12_1024": chains <= sms, "nr12_256": chains > sms}.get(cell, True), (cell, chains, sms)
    prob = _handle(mods, monkeypatch, _args(nr), E, env={"MPCMMD_INNER_CEM": mode} if mode else None, **SMALL)
    ora = O.OracleCEM(*_args(nr), **SMALL)
    b = episode_inputs(ora, E, 20 + nr + E)
    got = _launch(lambda: prob.solve_batch("mmd_opt", **b), want, cell)
    _check(got, ora, "mmd_opt", b, cell)
    _twins_differ(got, "mmd_opt", cell)


# ---------------------------------------------------------------------------------------------------------------------------------
# B3: grouped solve graphs (push_view offsets every per-episode array by the group's first episode)

def _auto_groups(sms, E, B):
    """solve_groups of csrc/mpcmmd_api.cu for mmd_opt with the fast inner kernel, restated"""
    chains = E * B
    if E < 2 or chains <= 6 * sms or chains > 36 * sms:
        return 1
    return min(3 if chains > 12 * sms else 2, E)


@gpu
@pytest.mark.parametrize("cost", ["cvar", "mmd_opt"])
def test_forced_groups_ragged(mods, monkeypatch, cost):
    """MPCMMD_GROUPS=3 at 7 episodes: groups of 2, 2 and 3 episodes on three graph branches; every episode equals its oracle solve"""
    _, O = mods
    E = 7
    prob = _handle(mods, monkeypatch, _args(), E, env={"MPCMMD_GROUPS": "3"}, **SMALL)
    ora = O.OracleCEM(*_args(), **SMALL)
    b = episode_inputs(ora, E, 30 + len(cost))
    want = {"k_inner_cem_lat<5, 0, 0, 0>"} if cost == "mmd_opt" else {"k_rollouts<2, false, 0, 0>"}
    got = _launch(lambda: prob.solve_batch(cost, **b), want, f"groups=3 {cost}")
    _check(got, ora, cost, b, f"groups=3 {cost}")


@gpu
@pytest.mark.parametrize("G", [2, 3])
def test_automatic_groups(mods, sms, monkeypatch, G):
    """the smallest mmd_opt batches of 100 samples that solve_groups splits into 2 and 3 groups: every episode equals the same episode
    solved alone, and the first and last episode of every group equal the oracle"""
    _, O = mods
    B = GROUPED["num_batch"]
    E = (6 if G == 2 else 12) * sms // B + 1
    assert _auto_groups(sms, E, B) == G
    prob = _handle(mods, monkeypatch, _args(), E, **GROUPED)
    one = _handle(mods, monkeypatch, _args(), 1, **GROUPED)
    ora = O.OracleCEM(*_args(), **GROUPED)
    b = episode_inputs(ora, E, 40 + G)
    got = prob.solve_batch("mmd_opt", **b)
    for e in range(E):
        solo = one.solve_batch("mmd_opt", **_sub(b, slice(e, e + 1)))
        for k in _keys("mmd_opt"):
            _eq(got[k][e], solo[k][0], f"{G} groups, {E} episodes: episode {e} {k} vs alone")
    edges = [i for gi in range(G) for i in (gi * E // G, (gi + 1) * E // G - 1)]
    _check(got, ora, "mmd_opt", b, f"{G} groups", edges + [2, 3])
    _twins_differ(got, "mmd_opt", f"{G} groups")


# ---------------------------------------------------------------------------------------------------------------------------------
# B4 / B5 / B6 / B7: large num_batch, sorted obstacle windows, wide reduced sets, Gaussian kernel

@gpu
@pytest.mark.parametrize("B", [1024, 1100])
def test_large_num_batch(mods, monkeypatch, B):
    """cvar at num_batch 1024 (rank-count selection with its largest key array) and 1100 (the 1024-thread k_noise / k_init / k_select)"""
    _, O = mods
    E, kw = 3, dict(num_batch=B, maxiter_cem=3)
    prob = _handle(mods, monkeypatch, _args(), E, **kw)
    ora = O.OracleCEM(*_args(), **kw)
    b = episode_inputs(ora, E, B)
    _check(prob.solve_batch("cvar", **b), ora, "cvar", b, f"B={B}")


def _fly_episodes(sms, nr):
    """episodes of 100 samples whose risk launch (episodes x 100 x nr rollouts) draws its controls on the fly"""
    return -(-2 * sms * ROLL_THREADS // (100 * nr)) + 1


@gpu
@pytest.mark.parametrize("size", ["staged", "fly"])
def test_sorted_windows(mods, sms, monkeypatch, size):
    """cvar with 32 obstacles: at 24 samples x 3 episodes k_rollouts<ROLL_STAGED> (plain obstacle loop), at enough 100-sample episodes
    k_rollouts<ROLL_FLY, SORTED>; the staged cell checks every episode, the fly cell episodes 0..3, the middle and the last"""
    _, O = mods
    args = _args(nobs=32)
    if size == "staged":
        E, kw, want, pick = 3, SMALL, {"k_rollouts<2, false, 0, 0>"}, None
    else:
        E, kw, want = _fly_episodes(sms, 5), dict(maxiter_cem=2), {"k_rollouts<1, true, 0, 0>"}
        pick = [0, 1, 2, 3, E // 2, E - 1]
    prob = _handle(mods, monkeypatch, args, E, **kw)
    ora = O.OracleCEM(*args, **kw)
    b = episode_inputs(ora, E, 50)
    got = _launch(lambda: prob.solve_batch("cvar", **b), want, f"32 obstacles {size}")
    _check(got, ora, "cvar", b, f"32 obstacles {size}", pick)


@gpu
@pytest.mark.parametrize("cost", ["cvar", "saa", "mmd_random"])
@pytest.mark.parametrize("nr", [65, 256])
def test_wide_reduced_sets(mods, wl, monkeypatch, cost, nr):
    """num_reduced 65 and 256: k_rollouts_wide against tests/wide_ref's solve, every episode"""
    _, O = mods
    E, kw = 3, dict(num_batch=24, maxiter_cem=3)
    args = _args(nr)
    prob = _handle(mods, monkeypatch, args, E, **kw)
    wide = W.WideOracle(O, wl, nr, *args[1:], **kw)
    b = episode_inputs(wide, E, nr + len(cost))
    got = _launch(lambda: prob.solve_batch(cost, **b), {"k_rollouts_wide<256, false, 0>"}, f"wide {cost} nr={nr}")
    refs = _pool(lambda e: wide.solve(cost, int(b["idx_mpc"][e]), b["init_state"][e], b["mean_param"][e], b["cov_param"][e],
                                      b["x_obs_traj"][e], b["y_obs_traj"][e], float(b["v_des"][e])), range(E))
    for e, ref in refs.items():
        for k in _keys(cost):
            _eq(got[k][e], ref[k], f"wide {cost} nr={nr} episode {e} {k}")


@gpu
@pytest.mark.parametrize("cost", ["mmd_opt", "mmd_random"])
def test_gaussian_kernel(mods, gk, monkeypatch, cost):
    """a kernel="gaussian" handle: every episode equals the kernel-form oracle (tests/gauss_oracle)"""
    from test_mmd_gaussian_kernel import KernelOracle
    _, O = mods
    E = 5
    prob = _handle(mods, monkeypatch, _args(), E, kernel="gaussian", **SMALL)
    ora = KernelOracle(O, gk, *_args(), kernel="gaussian", **SMALL)
    b = episode_inputs(ora, E, 60 + len(cost))
    want = {"k_inner_cem_lat<5, 0, 0, 1>"} if cost == "mmd_opt" else set()
    got = _launch(lambda: prob.solve_batch(cost, **b), want, f"gaussian kernel {cost}")
    _check(got, ora, cost, b, f"gaussian kernel {cost}")


# ---------------------------------------------------------------------------------------------------------------------------------
# C: full size, oracle-free

def _boundary(prob, out, b, what, tol=BC_TOL):
    """each plan's initial position, velocity and acceleration are its own episode's, and its final lateral velocity is 0"""
    P, Pd, Pdd = (np.asarray(a, np.float64) for a in (prob.P_jax, prob.Pdot_jax, prob.Pddot_jax))
    cx, cy = out["cx"].astype(np.float64), out["cy"].astype(np.float64)
    st = b["init_state"].astype(np.float64)
    got = np.stack([cx @ P[0], cx @ Pd[0], cx @ Pdd[0], cy @ P[0], cy @ Pd[0], cy @ Pdd[0], cy @ Pd[-1]], 1)
    want = np.concatenate([st[:, [0, 2, 4, 1, 3, 5]], np.zeros((len(st), 1))], 1)
    err = np.abs(got - want)
    assert np.isfinite(err).all() and err.max() <= tol, (what, np.unravel_index(np.argmax(err), err.shape), err.max())


@pytest.fixture(scope="module")
def full(mods):
    """the 200-episode batch at full CEM sizes, solved by cvar and mmd_opt on one handle"""
    cem_impl, O = mods
    prob = cem_impl.CEM(*FULL_ARGS, max_episodes=200)
    b = episode_inputs(O.OracleCEM(*FULL_ARGS), 200, 7)
    return prob, b, {c: prob.solve_batch(c, **b) for c in ("cvar", "mmd_opt")}


@gpu
@pytest.mark.parametrize("cost", ["cvar", "mmd_opt"])
def test_full_size_permutation(mods, full, cost):
    """200 episodes at full size, then the same episodes in a fixed permutation on the same handle: the outputs are permuted bit for bit;
    cvar episodes 0 (driver defaults), 1 (heading) and 199 and mmd_opt episode 1 equal the oracle; every plan meets its boundary conditions"""
    _, O = mods
    prob, b, out = full
    perm = np.random.default_rng(5).permutation(200)
    got = prob.solve_batch(cost, **_sub(b, perm))
    for k in _keys(cost):
        _eq(got[k], out[cost][k][perm], f"{cost} permuted {k}")
    _check(out[cost], O.OracleCEM(*FULL_ARGS), cost, b, f"full size {cost}", [0, 1, 199] if cost == "cvar" else [1])
    _boundary(prob, out[cost], b, f"{cost} exact projection")


@gpu
@pytest.mark.parametrize("E", [13, 25])
def test_full_size_permutation_grouped(mods, sms, full, E):
    """13 and 25 mmd_opt episodes (the automatic 2- and 3-group graphs on 148 SMs), in order and permuted: permuted bit for bit, and each
    episode equal to the same episode of the 200-episode solve"""
    prob, b, out = full
    sub = _sub(b, slice(0, E))
    got = prob.solve_batch("mmd_opt", **sub)
    perm = np.random.default_rng(E).permutation(E)
    pg = prob.solve_batch("mmd_opt", **_sub(sub, perm))
    for k in _keys("mmd_opt"):
        _eq(got[k], out["mmd_opt"][k][:E], f"{E} episodes ({_auto_groups(sms, E, 100)} groups) vs 200 {k}")
        _eq(pg[k], got[k][perm], f"{E} episodes permuted {k}")


@gpu
def test_full_size_tensor_core_projection(mods, monkeypatch, full):
    """MPCMMD_PROJ=tc-always on the 200-episode batch: every plan meets its own boundary conditions, its cx[:3] / cy[:3] are within 1e-5
    of the exact projection's (its trajectories are not bit-comparable, see test_solve_with_tensor_core_projection), and a permuted batch
    gives permuted outputs bit for bit"""
    prob0, b, out = full
    prob = _handle(mods, monkeypatch, FULL_ARGS, 200, env={"MPCMMD_PROJ": "tc-always"})
    perm = np.random.default_rng(9).permutation(200)
    for cost in ("cvar", "mmd_opt"):
        t = prob.solve_batch(cost, **b)
        _boundary(prob, t, b, f"{cost} tensor-core projection")
        np.testing.assert_allclose(t["cx"][:, :3], out[cost]["cx"][:, :3], rtol=1e-5, atol=1e-5, err_msg=cost)
        np.testing.assert_allclose(t["cy"][:, :3], out[cost]["cy"][:, :3], rtol=1e-5, atol=1e-5, err_msg=cost)
        tp = prob.solve_batch(cost, **_sub(b, perm))
        for k in _keys(cost):
            _eq(tp[k], t[k][perm], f"{cost} tensor-core projection, permuted {k}")


# ---------------------------------------------------------------------------------------------------------------------------------
# D: one handle across batches of different content and size

REUSE = {
    # cell: (num_reduced, cost, MPCMMD_INNER_CEM)
    "cvar": (5, "cvar", None),
    "mmd_opt_fast": (5, "mmd_opt", "cta"),
    "mmd_opt_generic": (5, "mmd_opt", "generic"),
    "wide_cvar": (65, "cvar", None),
}


def _poisoned(b):
    """episode 1 with NaN obstacle coordinates, episode 2 with a covariance that is not positive definite, episode 3 at rest"""
    b = {n: v.copy() for n, v in b.items()}
    b["x_obs_traj"][1, 0, 10:30] = np.nan; b["y_obs_traj"][1, 1, 40] = np.nan
    b["cov_param"][2, 2, 2] = -1.0
    b["init_state"][3, 2:4] = 0.0
    return b


@gpu
@pytest.mark.parametrize("cell", list(REUSE))
def test_handle_reuse(mods, monkeypatch, cell):
    """on one handle: a poisoned batch of 5, a clean batch of 5, 3 episodes, then 7 episodes of new inputs; each call equals the same call
    on a fresh handle (solve graphs are cached per (cost, episodes); multipliers, slacks, risk and output scratch persist between solves)"""
    _, O = mods
    nr, cost, mode = REUSE[cell]
    args, env = _args(nr), {"MPCMMD_INNER_CEM": mode} if mode else None
    kw = SMALL if nr <= 64 else dict(num_batch=24, maxiter_cem=3)
    ora = O.OracleCEM(*_args(), **SMALL)
    clean = episode_inputs(ora, 5, 70)
    calls = [("poisoned", _poisoned(clean)), ("clean", clean), ("3 episodes", _sub(clean, slice(1, 4))), ("7 new", episode_inputs(ora, 7, 71))]
    prob = _handle(mods, monkeypatch, args, 7, env=env, **kw)
    for what, b in calls:
        got = prob.solve_batch(cost, **b)
        fresh = _handle(mods, monkeypatch, args, len(b["idx_mpc"]), env=env, **kw)
        _same(got, fresh.solve_batch(cost, **b), cost, f"{cell} {what}: reused vs fresh handle")
        del fresh
    assert np.isfinite(got["cx"]).all()


# ---------------------------------------------------------------------------------------------------------------------------------
# E: the CUDA-tensor entry point on torch streams

@gpu
def test_device_path_on_streams(mods, monkeypatch):
    """solve_batch_device with CUDA-tensor inputs on a non-default torch stream equals solve_batch; a cvar and an mmd_opt handle enqueued
    on two streams before one synchronize equal their results solved one after the other"""
    import torch
    _, O = mods
    E = 5
    ora = O.OracleCEM(*_args(), **SMALL)
    b = {c: episode_inputs(ora, E, 80 + len(c)) for c in ("cvar", "mmd_opt")}
    probs = {c: _handle(mods, monkeypatch, _args(), E, **SMALL) for c in ("cvar", "mmd_opt")}
    host = {c: probs[c].solve_batch(c, **b[c]) for c in probs}
    _check(host["mmd_opt"], ora, "mmd_opt", b["mmd_opt"], "host path")
    streams = {c: torch.cuda.Stream() for c in probs}
    outs = {}
    for c in probs:
        with torch.cuda.stream(streams[c]):
            tin = {k: torch.as_tensor(v, device="cuda") for k, v in b[c].items()}
            outs[c] = probs[c].solve_batch_device(c, **tin)
    torch.cuda.synchronize()
    for c in probs:
        _same({k: v.cpu().numpy() for k, v in outs[c].items() if k != "_keepalive"}, host[c], c, f"{c}: device path on its own stream")
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        tin = {k: torch.as_tensor(v, device="cuda") for k, v in b["cvar"].items()}
        one = probs["cvar"].solve_batch_device("cvar", **tin)
    s.synchronize()
    _same({k: v.cpu().numpy() for k, v in one.items() if k != "_keepalive"}, host["cvar"], "cvar", "cvar: device path alone")


# ---------------------------------------------------------------------------------------------------------------------------------
# F: Monte-Carlo validation with per-plan initial states

def _plans(group, seed):
    """the golden plans of one group, each item given its own initial state (y0 within 0.45 of the start lane, vx, vy, heading)"""
    from test_validation import _case_inputs, _cases, _fake_prob, _items
    g, names = _cases()
    names = [n for n in names if n.startswith(group)]
    items = _items(g, names)
    rng = np.random.default_rng(seed)
    for i, it in enumerate(items):
        s = np.array(it["init_state"], np.float64)
        s[1] += rng.uniform(-0.45, 0.45); s[2] = rng.uniform(3.0, 8.0); s[3] = rng.uniform(-0.6, 0.6)
        it["init_state"] = s
    prob = _fake_prob("static" if group.startswith("S_") else "dynamic", g[names[0] + "_args"])
    return g, names, items, prob, [_case_inputs(g, n) for n in names]


@gpu
@pytest.mark.parametrize("group", ["S_beta", "S_gauss", "D_gauss"])
def test_validation_per_plan_states(mods, group):
    """compute_stats_batch and risk_stats_batch(rng="host") on plans with distinct initial states: the counts of every plan equal the
    oracle's compute_stats from that plan's own state; rng="jax" counts equal mpcmmd_validate_host on the restated controls"""
    from mpcmmd_b200 import binding as B, validation as V
    from oracle import oracle_validation as OV
    from test_validation_jax_rng import _restated, _validate_host
    g, names, items, prob, cases = _plans(group, 90 + len(group))
    variant, c, num_obs, noise_level, num_prime, noise, _, _, _ = cases[0]
    count, lane = V.compute_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, device=0)
    risk = V.risk_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, device=0)
    want, moved = [], 0
    for i, (it, cs) in enumerate(zip(items, cases)):
        xt, yt = cs[7], cs[8]
        co, lo, _, _ = OV.compute_stats(c, it["cx"], it["cy"], it["init_state"], xt, yt, num_prime, noise_level, noise, it["key"],
                                        obs_f32=(variant == "static"))
        want.append((co, lo))
        if i and (co, lo) != OV.compute_stats(c, it["cx"], it["cy"], items[0]["init_state"], xt, yt, num_prime, noise_level, noise, it["key"],
                                              obs_f32=(variant == "static"))[:2]:
            moved += 1
    assert moved, f"{group}: no plan's counts depend on its initial state"
    assert [(int(a), int(b_)) for a, b_ in zip(count, lane)] == want, (group, count, lane, want)
    assert [(int(a), int(b_)) for a, b_ in zip(risk["count"], risk["count_lane"])] == want, (group, risk["count"], risk["count_lane"], want)
    jc, jl = V.compute_stats_batch(prob, items, num_prime, noise_level, noise, num_obs, device=0, rng="jax")
    a_r, s_r = _restated(V, prob, items, num_prime, num_obs, noise_level, noise, 1000)
    hc, hl = _validate_host(V, B, prob, items, num_prime, num_obs, a_r, s_r)
    assert np.array_equal(jc, hc) and np.array_equal(jl, hl), (group, jc, hc, jl, hl)
