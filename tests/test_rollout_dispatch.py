"""Every instantiation of the rollout family against the oracle, each cell checked by the name of the kernel it launched.

launch_risk (csrc/mpcmmd_api.cu) picks the rollout kernel from the launch's size as well as from its configuration: cvar / saa / mmd_random
stage their controls (k_rollouts<ROLL_STAGED>, plain obstacle loop) while n_samples * num_reduced < 2 * SMs * ROLL_THREADS and draw them on
the fly above that (k_rollouts<ROLL_FLY>), and only ROLL_FLY, k_rollouts_wide and k_opt_risk have SORTED builds: the binary search over the
per-knot sorted obstacle lists used when num_obs > OBS_SORT_MIN (8).  mmd_opt picks one of three bodies (plain, write, fold) from the chain
count, num_reduced and num_obs.  A test written at a convenient size can therefore run a different kernel from the one it describes, so
every cell here states the instantiation(s) it reaches and asserts them from torch.profiler's kernel records, and a CPU test holds the
table of cells to the instantiations the library actually contains.  Launch sizes come from the SM count.

Templates: k_rollouts<MODE, SORTED, NZ, OV> (MODE 0 ROLL_OPT, 1 ROLL_FLY, 2 ROLL_STAGED; NZ 0 Gaussian, 1 Beta candidate table, 2 run-time
choice: injected draws, direct sampler or the table; OV 0 plain, 1 write, 2 fold), k_rollouts_wide<256, SORTED, NZ>, k_opt_risk<SORTED>.

The sorted cells run edge scenes built from the oracle's own rollouts of sample 0: at every knot t < num_prime obstacles sit ahead of the
front-most and behind the rear-most of these rollouts -- one just inside the ellipse ahead (|dx| = a_obs - 0.005: the largest obstacle cost
sample 0 meets, which a window narrower by 0.01 m would miss), others at |dx| = a_obs and one ulp either side, at the window half-width
obs_win and one ulp either side, three with equal x, and at +-inf x or y -- while the remaining obstacles move across the vehicle's path off the road, overtaking each other, so the sorted order changes
from knot to knot.  Variants: NaN x at some knots and NaN y at others (the per-knot obs_nan fallback to the plain loop), and a vehicle that
drives past x = 1e4 (where the window is not used).  NaN vehicle states come from NaN Beta draws through mpcmmd_stage_risk_injected."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import kernel_names as KN
import wide_ref as W

gpu = pytest.mark.gpu
f32 = np.float32
ROLL_THREADS = 128                                                    # k_rollouts CTA size (csrc/k_risk.cuh)
A_OBS = 4.25
OBS_WIN = f32(np.sqrt(np.float64(f32(A_OBS ** 2))) * (1.0 + 1e-6) + 1.0e-2)      # DCfg::obs_win (csrc/mpcmmd_api.cu)
ST0 = np.array([0.0, 1.75, 5.0, 0.0, 0.0], f32)
ST0_FAR = np.array([1.0e4 - 8.0, 1.75, 5.0, 0.0, 0.0], f32)      # the rollouts pass x = 1e4 within the horizon
INNER = dict(num_samples_cem=40, maxiter_beta_cem=3)
SMALL = dict(num_batch=24, maxiter_cem=3, num_samples_cem=40, maxiter_beta_cem=3)
FIELDS = ("risk", "lane", "beta", "sigma", "res_beta")
NZ_NAME = {"gaussian": 0, "beta": 2, "injected": 2}                 # NZ of a stage launch: the stage entry points have no candidate table

# ---------------------------------------------------------------------------------------------------------------------------------
# instantiation -> the cells below that launch it (and assert it by name)

TABLE = {
    "k_rollouts<0, false, 0, 0>": ["opt_sorted_stage/gaussian"],
    "k_rollouts<0, false, 1, 0>": ["opt_plain_solve/beta"],
    "k_rollouts<0, false, 2, 0>": ["opt_sorted_stage/beta"],
    "k_rollouts<0, false, 0, 1>": ["opt_write_stage/gaussian"],
    "k_rollouts<0, false, 1, 1>": ["opt_write_solve/beta"],
    "k_rollouts<0, false, 2, 1>": ["opt_write_stage/beta"],
    "k_rollouts<0, false, 0, 2>": ["opt_fold_stage/gaussian"],
    "k_rollouts<0, false, 1, 2>": ["opt_fold_solve/beta"],
    "k_rollouts<0, false, 2, 2>": ["opt_fold_stage/beta"],
    "k_rollouts<1, false, 0, 0>": ["fly_stage/gaussian"],
    "k_rollouts<1, false, 1, 0>": ["fly_solve/beta"],
    "k_rollouts<1, false, 2, 0>": ["fly_stage/beta"],
    "k_rollouts<1, true, 0, 0>": ["fly_sorted_stage/gaussian", "fly_sorted_solve/gaussian"],
    "k_rollouts<1, true, 2, 0>": ["fly_sorted_stage/beta", "fly_sorted_stage/injected", "fly_sorted_solve/beta"],
    "k_rollouts<2, false, 0, 0>": ["staged_stage/gaussian"],
    "k_rollouts<2, false, 1, 0>": ["staged_solve/beta"],
    "k_rollouts<2, false, 2, 0>": ["staged_stage/beta"],
    "k_rollouts_wide<256, false, 0>": ["wide_stage/gaussian"],
    "k_rollouts_wide<256, false, 1>": ["wide_solve/beta"],
    "k_rollouts_wide<256, false, 2>": ["wide_stage/beta"],
    "k_rollouts_wide<256, true, 0>": ["wide_sorted_stage/gaussian", "wide_sorted_solve/gaussian"],
    "k_rollouts_wide<256, true, 1>": ["wide_sorted_solve/beta"],
    "k_rollouts_wide<256, true, 2>": ["wide_sorted_stage/beta", "wide_sorted_stage/injected"],
    "k_opt_risk<false>": ["opt_fold_stage/gaussian", "opt_fold_stage/beta", "opt_fold_solve/beta"],
    "k_opt_risk<true>": ["opt_sorted_stage/gaussian", "opt_sorted_stage/beta", "opt_plain_solve/beta"],
}


def _want(cell):
    return {k for k, cells in TABLE.items() if cell in cells}


def _launch(cell, fn):
    """fn() under the profiler; asserts that every instantiation TABLE assigns to `cell` ran, and returns fn's result"""
    out, names = KN.launched(fn)
    ran = KN.family(names)
    missing = _want(cell) - ran
    assert not missing, f"{cell}: expected {sorted(_want(cell))} to run, the profiler saw {sorted(ran)} (all kernels: {sorted(names)})"
    return out


# ---------------------------------------------------------------------------------------------------------------------------------
# helpers

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
def sms(mods):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture(scope="module")
def wl(mods, tmp_path_factory):
    return W.build_lib(tmp_path_factory.mktemp("wide_oracle"))


def _fly_threshold(sms):
    """rollouts of the smallest launch that draws its controls on the fly (roll_stage_ctrl of csrc/mpcmmd_api.cu)"""
    return 2 * sms * ROLL_THREADS


def _fly_samples(sms, nr):
    return -(-_fly_threshold(sms) // nr) + 7


def _controls(ora, rng, n, bases=12):
    """n control sequences: `bases` projected ones, each sample a randomly scaled copy of one of them"""
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
    pick[0] = 0
    return ((acc[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32), (steer[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32))


def _pool(fn, idx):
    idx = [int(i) for i in idx]
    with ThreadPoolExecutor(max_workers=max(1, min(len(idx), os.cpu_count() or 1))) as ex:
        return dict(zip(idx, ex.map(fn, idx)))


def _check(got, refs, fields, what):
    for i, ref in refs.items():
        for k in fields:
            _eq(got[k][i], ref[k], f"{what} sample {i} {k}")


def _fields(cost):
    return FIELDS if cost == "mmd_opt" else ("risk", "lane", "beta", "sigma") if cost == "mmd_random" else ("risk", "lane")


def _ulp(x, d):
    return np.nextafter(f32(x), f32(np.inf) if d > 0 else f32(-np.inf))


def edge_scene(xr, yr, num_prime, nobs, kind="edge", seed=0):
    """(x_obs, y_obs) (nobs, 100) around the recorded points xr, yr (R, num_prime) of a sample's rollouts: see the module docstring"""
    rng = np.random.default_rng(seed)
    R = xr.shape[0]
    t = np.linspace(0.0, 15.0, 100).astype(f32)
    base = float(xr[0, 0])
    x0 = rng.uniform(base - 10.0, base + 110.0, nobs); vx = rng.uniform(-4.0, 12.0, nobs)
    xo = (x0[:, None] + vx[:, None] * t[None]).astype(f32)
    yo = np.repeat((rng.choice([-1.0, 1.0], nobs) * rng.uniform(6.0, 10.0, nobs))[:, None], 100, 1).astype(f32)
    for k in range(num_prime):
        fin = np.flatnonzero(np.isfinite(xr[:, k]) & np.isfinite(yr[:, k]))
        if fin.size == 0:
            continue
        hi, lo = fin[np.argmax(xr[fin, k])], fin[np.argmin(xr[fin, k])]
        x, y = f32(xr[hi, k]), f32(yr[hi, k])              # ahead of the front-most rollout: every other rollout is farther away
        xb, yb = f32(xr[lo, k]), f32(yr[lo, k])            # behind the rear-most one
        a, w = f32(x + f32(A_OBS)), f32(x + OBS_WIN)
        ab, wb = f32(xb - f32(A_OBS)), f32(xb - OBS_WIN)
        eq = f32(x + f32(A_OBS - 0.003))
        special = [(a, y), (_ulp(a, 1), y), (_ulp(a, -1), y), (ab, yb), (_ulp(ab, 1), yb), (_ulp(ab, -1), yb),
                   (w, y), (_ulp(w, 1), y), (_ulp(w, -1), y), (wb, yb), (_ulp(wb, 1), yb), (_ulp(wb, -1), yb),
                   (eq, y), (eq, f32(y + 0.4)), (eq, f32(y - 9.0)),
                   (f32(np.inf), y), (f32(-np.inf), y), (f32(x + 1.0), f32(np.inf)), (f32(x - 1.0), f32(-np.inf))]
        m = min(len(special), nobs - 3)
        pick = [(f32(x + f32(A_OBS - 0.005)), y)] + [special[(3 * k + j) % len(special)] for j in range(m)]
        slots = rng.permutation(nobs)[:len(pick)]
        for o, (px, py) in zip(slots, pick):
            xo[o, k] = px; yo[o, k] = py
    if kind == "nan":
        for k in range(1, num_prime, 7):
            xo[rng.integers(nobs), k] = np.nan
        for k in range(4, num_prime, 7):
            yo[rng.integers(nobs), k] = np.nan
    return np.ascontiguousarray(xo), np.ascontiguousarray(yo)


def _rollouts(ora, cost, acc0, steer0, st0, noise_t, beta_draws=None):
    """recorded points (R, num_prime) of sample 0's rollouts, from the oracle"""
    xo = np.full((ora.num_obs, 100), 1.0e3, f32); yo = np.zeros((ora.num_obs, 100), f32)
    r = ora.risk(cost, acc0, steer0, st0, noise_t, xo, yo, want_rollouts=True, beta_draws=beta_draws)
    return r["x_roll"], r["y_roll"]


def _assert_far(xr):
    ax = np.abs(xr[np.isfinite(xr)])
    assert (ax >= 1.0e4).any() and (ax < 1.0e4).any(), "the far scene's rollouts do not cross |x| = 1e4"


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: the table covers exactly the instantiations the library holds

FLY_CASES = ([(c, nobs, nz, "edge") for c in ("cvar", "saa", "mmd_random") for nobs in (9, 32, 64) for nz in ("gaussian", "beta")]
             + [("cvar", 32, "gaussian", "nan"), ("cvar", 32, "beta", "far"), ("saa", 9, "beta", "nan"), ("mmd_random", 64, "gaussian", "far"),
                ("cvar", 64, "injected", "edge"), ("mmd_random", 32, "injected", "edge"), ("saa", 9, "injected", "far"),
                ("cvar", 32, "injected", "nan")])
OPT_CASES = [(nz, scene) for nz in ("gaussian", "beta") for scene in ("edge", "nan", "far")]
WIDE_CASES = ([(c, nr, nobs, nz, "edge") for c in ("cvar", "saa", "mmd_random") for nr in (65, 256, 1024) for nobs in (9, 64)
               for nz in ("gaussian", "beta", "injected")]
              + [("cvar", 256, 64, "injected", "nan"), ("mmd_random", 65, 9, "injected", "far"), ("saa", 1024, 64, "gaussian", "nan"),
                 ("cvar", 65, 64, "gaussian", "far")])
SOLVE_NOISES = ("gaussian", "beta")
OTHER_CELLS = {
    # cell: (kind, cost, num_reduced, num_obs, noise)
    "opt_fold_stage/gaussian": ("stage", "mmd_opt", 5, 2, "gaussian"),
    "opt_fold_stage/beta": ("stage", "mmd_opt", 5, 2, "beta"),
    "opt_fold_solve/beta": ("solve", "mmd_opt", 5, 2, "beta"),
    "opt_plain_solve/beta": ("solve", "mmd_opt", 5, 9, "beta"),
    "opt_write_stage/gaussian": ("stage", "mmd_opt", 6, 2, "gaussian"),
    "opt_write_stage/beta": ("stage", "mmd_opt", 6, 2, "beta"),
    "opt_write_solve/beta": ("solve", "mmd_opt", 6, 2, "beta"),
    "staged_stage/gaussian": ("stage", "cvar", 5, 2, "gaussian"),
    "staged_stage/beta": ("stage", "cvar", 5, 2, "beta"),
    "staged_solve/beta": ("solve", "cvar", 5, 2, "beta"),
    "fly_stage/gaussian": ("fly_stage", "cvar", 5, 2, "gaussian"),
    "fly_stage/beta": ("fly_stage", "cvar", 5, 2, "beta"),
    "fly_solve/beta": ("fly_solve", "cvar", 5, 4, "beta"),
    "wide_stage/gaussian": ("stage", "cvar", 65, 2, "gaussian"),
    "wide_stage/beta": ("stage", "saa", 65, 2, "beta"),
    "wide_solve/beta": ("solve", "cvar", 65, 2, "beta"),
}


def _cell_keys():
    keys = {f"fly_sorted_stage/{nz}" for _, _, nz, _ in FLY_CASES}
    keys |= {f"opt_sorted_stage/{nz}" for nz, _ in OPT_CASES}
    keys |= {f"wide_sorted_stage/{nz}" for _, _, _, nz, _ in WIDE_CASES}
    keys |= {f"{p}/{nz}" for p in ("fly_sorted_solve", "wide_sorted_solve") for nz in SOLVE_NOISES}
    return keys | set(OTHER_CELLS)


def test_instantiation_table_matches_library(built):
    """the rollout-family instantiations in libmpcmmd.so are exactly TABLE's keys, and every cell TABLE names is one of this module's cells"""
    have = KN.built_instantiations(built.LIB)
    assert len(have) == 25, sorted(have)
    assert have == set(TABLE), f"in the library but not in TABLE: {sorted(have - set(TABLE))}; in TABLE but not built: {sorted(set(TABLE) - have)}"
    named = {c for cells in TABLE.values() for c in cells}
    assert named <= _cell_keys(), sorted(named - _cell_keys())
    assert all(TABLE.values())


def test_edge_scene_places_the_edges():
    """the scene builder puts, at knot k, obstacles exactly a_obs and obs_win ahead of the front-most / behind the rear-most rollout, one ulp
    either side, and one just inside the ellipse ahead"""
    rng = np.random.default_rng(1)
    xr = np.cumsum(rng.uniform(0.5, 2.0, (5, 30)), 1).astype(f32); yr = rng.uniform(1.0, 2.5, (5, 30)).astype(f32)
    xo, yo = edge_scene(xr, yr, 30, 64)
    for k in range(30):
        x, xb = f32(xr[:, k].max()), f32(xr[:, k].min())
        col = set(xo[:, k].tolist())
        assert f32(x + f32(A_OBS - 0.005)) in col, k
        for v in (f32(x + f32(A_OBS)), f32(xb - f32(A_OBS)), f32(x + OBS_WIN), f32(xb - OBS_WIN)):
            assert {v, _ulp(v, 1), _ulp(v, -1)} <= col, (k, v)
        assert np.isinf(xo[:, k]).sum() == 2 and np.isinf(yo[:, k]).sum() == 2
    xo9, _ = edge_scene(xr, yr, 30, 9)
    assert np.isfinite(xo9[:, 30:]).all()
    xn, yn = edge_scene(xr, yr, 30, 32, "nan")
    assert np.isnan(xn).any(axis=0).sum() == len(range(1, 30, 7)) and np.isnan(yn).any(axis=0).sum() == len(range(4, 30, 7))


# ---------------------------------------------------------------------------------------------------------------------------------
# ROLL_FLY, sorted windows: stages just above the threshold

def _beta_draws(rng, n, n_el, nan_samples=()):
    b1 = rng.beta(2.0, 5.0, (n, n_el)).astype(f32); b2 = rng.beta(2.0, 5.0, (n, n_el)).astype(f32)
    for s in nan_samples:                              # a NaN draw mid-horizon: the rollout's state is NaN from there on
        b1[s, (7 * s) % n_el] = np.nan
        b2[s, (11 * s + 3) % n_el] = np.nan
    return b1, b2


@gpu
@pytest.mark.parametrize("cost,nobs,noise,scene", FLY_CASES)
def test_fly_sorted_stage(mods, sms, cost, nobs, noise, scene):
    """a launch just above the staging threshold runs k_rollouts<ROLL_FLY, SORTED>; every cvar / saa sample (a strided subset of mmd_random)
    equals the oracle, and the whole launch equals the same samples run as launches small enough to stage their controls (plain obstacle loop)"""
    cem_impl, O = mods
    nr, np_ = 5, 30
    n = _fly_samples(sms, nr)
    assert n * nr >= _fly_threshold(sms) and (n // 2 + 1) * nr < _fly_threshold(sms)
    args = (nr, nobs, 0.1 if noise == "gaussian" else 0.3, np_, "gaussian" if noise == "gaussian" else "beta", 0.05, 0.01)
    prob = cem_impl.CEM(*args, max_episodes=-(-n // 100)); ora = O.OracleCEM(*args)
    rng = np.random.default_rng(100 * nobs + len(cost))
    acc, steer = _controls(ora, rng, n)
    st0 = ST0_FAR if scene == "far" else ST0
    noise_t = ora.noise_tables(4242, 3)
    draws = _beta_draws(rng, n, nr * np_, nan_samples=range(1, n, 97)) if noise == "injected" else None
    xr, yr = _rollouts(ora, cost, acc[0], steer[0], st0, noise_t, None if draws is None else (draws[0][0], draws[1][0]))
    if scene == "far":
        _assert_far(xr)
    xo, yo = edge_scene(xr, yr, np_, nobs, scene, seed=nobs)
    if noise == "injected":
        got = _launch("fly_sorted_stage/injected", lambda: prob.stage_risk_injected(cost, acc, steer, st0, noise_t[2], draws[0], draws[1], xo, yo))
        half = n // 2 + 1
        parts = [prob.stage_risk_injected(cost, acc[a:a + half], steer[a:a + half], st0, noise_t[2], draws[0][a:a + half], draws[1][a:a + half], xo, yo)
                 for a in range(0, n, half)]
    else:
        got = _launch(f"fly_sorted_stage/{noise}", lambda: prob.stage_risk(cost, acc, steer, st0, noise_t, xo, yo))
        half = n // 2 + 1
        parts, names = KN.launched(lambda: [prob.stage_risk(cost, acc[a:a + half], steer[a:a + half], st0, noise_t, xo, yo) for a in range(0, n, half)])
        assert f"k_rollouts<2, false, {NZ_NAME[noise]}, 0>" in KN.family(names)
    staged = {k: np.concatenate([p[k] for p in parts]) for k in parts[0]}
    for k in _fields(cost):
        _eq(got[k], staged[k], f"{cost} {nobs} {noise} {scene} {k}: one ROLL_FLY launch of {n} vs ROLL_STAGED launches of {half}")
    idx = range(n) if cost != "mmd_random" else sorted(set(range(0, n, 41)) | {n - 1})
    refs = _pool(lambda i: ora.risk(cost, acc[i], steer[i], st0, noise_t, xo, yo,
                                    beta_draws=None if draws is None else (draws[0][i], draws[1][i])), idx)
    _check(got, refs, _fields(cost), f"{cost} nobs={nobs} {noise} {scene}")
    if scene == "nan":                                 # every rollout passes a NaN knot: its cost is NaN (cvar / saa then count no tail / no hit)
        assert np.isnan(refs[0]["red_cost"]).all()
    elif noise != "injected":
        assert np.isfinite(got["risk"]).all() and (got["risk"][0] != 0 or cost != "cvar")
    if cost == "cvar" and scene != "nan":
        assert np.any(got["risk"] != got["risk"][0])


# ---------------------------------------------------------------------------------------------------------------------------------
# mmd_opt: k_opt_risk<true> re-rolls the chosen reduced set with sorted windows

@gpu
@pytest.mark.parametrize("noise,scene", OPT_CASES)
def test_opt_sorted_stage(mods, noise, scene):
    """mmd_opt at 32 obstacles: the plain ROLL_OPT body (no fold above 8 obstacles), the inner CEM, then k_opt_risk<true>; the scene is built
    around every mother rollout of sample 0, so whichever reduced set the inner CEM chooses re-rolls through the edges"""
    cem_impl, O = mods
    nr, np_, nobs, n = 5, 30, 32, 6
    args = (nr, nobs, 0.1 if noise == "gaussian" else 0.3, np_, noise, 0.05, 0.01)
    prob = cem_impl.CEM(*args, max_episodes=1, **INNER); ora = O.OracleCEM(*args, **INNER)
    rng = np.random.default_rng(77)
    acc, steer = _controls(ora, rng, n)
    st0 = ST0_FAR if scene == "far" else ST0
    noise_t = ora.noise_tables(91, 4)
    xr, yr = _rollouts(ora, "mmd_opt", acc[0], steer[0], st0, noise_t)
    assert xr.shape[0] == nr * nr
    if scene == "far":
        _assert_far(xr)
    xo, yo = edge_scene(xr, yr, np_, nobs, scene, seed=5)
    got = _launch(f"opt_sorted_stage/{noise}", lambda: prob.stage_risk("mmd_opt", acc, steer, st0, noise_t, xo, yo))
    refs = _pool(lambda i: ora.risk("mmd_opt", acc[i], steer[i], st0, noise_t, xo, yo), range(n))
    _check(got, refs, FIELDS, f"mmd_opt {noise} {scene}")
    if scene == "nan":
        assert np.isnan(got["risk"]).all() and np.isnan(refs[0]["red_cost"]).all()


# ---------------------------------------------------------------------------------------------------------------------------------
# k_rollouts_wide, sorted windows

@gpu
@pytest.mark.parametrize("cost,nr,nobs,noise,scene", WIDE_CASES)
def test_wide_sorted_stage(mods, wl, cost, nr, nobs, noise, scene):
    """num_reduced 65..1024 with more than 8 obstacles: k_rollouts_wide<256, true, NZ> against tests/wide_ref.  The scene is built from the
    first five rollouts of sample 0, which the nr-5 oracle rolls out bit for bit when the Beta draws and z3 are injected (for the Gaussian
    and direct-sampler cells the same scene is near, not at, the edges); the injected cells also give samples 3..5 NaN draws"""
    cem_impl, O = mods
    np_, n = 20, 6
    beta = noise != "gaussian"
    args = (nobs, 0.3 if beta else 0.1, np_, "beta" if beta else "gaussian", 0.05, 0.01)
    prob = cem_impl.CEM(nr, *args, max_episodes=1); wide = W.WideOracle(O, wl, nr, *args); ora5 = O.OracleCEM(5, *args)
    rng = np.random.default_rng(nr + nobs)
    acc, steer = _controls(wide, rng, n)
    st0 = ST0_FAR if scene == "far" else ST0
    noise_t = wide.noise_tables(17, 2)
    z3_5 = ora5.noise_tables(17, 2)[2]
    z3 = np.concatenate([z3_5, rng.normal(0, 1, nr * np_ - z3_5.size).astype(f32)])
    b1, b2 = _beta_draws(rng, n, nr * np_, nan_samples=(3, 4, 5))
    n5 = 5 * np_
    xr, yr = _rollouts(ora5, "cvar", acc[0], steer[0], st0, (z3_5, z3_5, z3_5, None, [0, 0, 0, 0]),
                       beta_draws=(b1[0, :n5].reshape(5, np_), b2[0, :n5].reshape(5, np_)))
    if scene == "far":
        _assert_far(xr)
    xo, yo = edge_scene(xr, yr, np_, nobs, scene, seed=nr)
    if noise == "injected":
        got = _launch("wide_sorted_stage/injected", lambda: prob.stage_risk_injected(cost, acc, steer, st0, z3, b1, b2, xo, yo))
        inj_t = (z3, z3, z3, None, [0, 0, 0, 0])
        refs = _pool(lambda i: wide.risk(cost, acc[i], steer[i], st0, inj_t, xo, yo, beta_draws=(b1[i], b2[i])), range(n))
        assert all(np.isnan(refs[i]["red_cost"]).any() for i in (3, 4, 5))
    else:
        got = _launch(f"wide_sorted_stage/{noise}", lambda: prob.stage_risk(cost, acc, steer, st0, noise_t, xo, yo))
        refs = _pool(lambda i: wide.risk(cost, acc[i], steer[i], st0, noise_t, xo, yo), range(n))
    _check(got, refs, _fields(cost), f"{cost} nr={nr} nobs={nobs} {noise} {scene}")
    if scene == "nan":
        assert all(np.isnan(refs[i]["red_cost"]).all() for i in range(n))


# ---------------------------------------------------------------------------------------------------------------------------------
# full solves with sorted windows

def _batch(O, ora, E, nobs):
    from mpcmmd_b200 import scenes
    eps = [O.static_episode(nobs, k) if nobs <= 9 else scenes.scaled_scene(nobs, k) for k in range(E)]
    tr = [ora.compute_obs_trajectories(*sc) for sc, _ in eps]
    init_state, mean, cov, v_des = O.driver_inputs("static")
    return dict(idx_mpc=[i for _, i in eps], init_state=np.stack([init_state] * E), mean_param=np.stack([mean] * E),
                cov_param=np.stack([cov] * E), x_obs_traj=np.stack([t[0] for t in tr]), y_obs_traj=np.stack([t[1] for t in tr]), v_des=[v_des] * E)


def _ref_solve(ora, cost, b, e):
    return ora.solve(cost, b["idx_mpc"][e], b["init_state"][e], b["mean_param"][e], b["cov_param"][e], b["x_obs_traj"][e], b["y_obs_traj"][e],
                     b["v_des"][e])


def _solve_keys(cost):
    return ("cx", "cy", "cost_obs", "cost_lane") + (("beta", "sigma", "res_beta") if cost == "mmd_opt" else ())


def _fly_episodes(sms, nr):
    """episodes of 100 samples whose risk launch (episodes x 100 x nr rollouts) draws its controls on the fly"""
    return -(-_fly_threshold(sms) // (100 * nr)) + 1


@gpu
@pytest.mark.parametrize("noise", SOLVE_NOISES)
def test_fly_sorted_solve(mods, sms, noise):
    """cvar with 9 obstacles over enough episodes that every iteration's risk launch is ROLL_FLY with sorted windows: with beta noise this
    is the NZ_ANY build replaying the Beta candidate table.  Every episode equals the oracle's solve"""
    cem_impl, O = mods
    nr, nobs = 5, 9
    E = _fly_episodes(sms, nr)
    kw = dict(maxiter_cem=2)
    args = (nr, nobs, 0.3 if noise == "beta" else 0.1, 30, noise, 0.02, 0.01)
    prob = cem_impl.CEM(*args, max_episodes=E, **kw); ora = O.OracleCEM(*args, **kw)
    b = _batch(O, ora, E, nobs)
    got = _launch(f"fly_sorted_solve/{noise}", lambda: prob.solve_batch("cvar", **b))
    refs = _pool(lambda e: _ref_solve(ora, "cvar", b, e), range(E))
    for e, ref in refs.items():
        for k in _solve_keys("cvar"):
            _eq(got[k][e], ref[k], f"cvar {noise} {E} episodes: episode {e} {k}")
    assert np.isfinite(got["cx"]).all()


@gpu
@pytest.mark.parametrize("noise", SOLVE_NOISES)
def test_wide_sorted_solve(mods, wl, noise):
    """cvar at num_reduced 128 with 9 obstacles: k_rollouts_wide<256, true, NZ> in the solve graph (the Beta candidate table with beta noise)"""
    cem_impl, O = mods
    E, nr = 2, 128
    args = (9, 0.3 if noise == "beta" else 0.1, 30, noise, 0.02, 0.01)
    prob = cem_impl.CEM(nr, *args, max_episodes=E, num_batch=24, maxiter_cem=3); wide = W.WideOracle(O, wl, nr, *args, num_batch=24, maxiter_cem=3)
    b = _batch(O, wide, E, 9)
    got = _launch(f"wide_sorted_solve/{noise}", lambda: prob.solve_batch("cvar", **b))
    for e in range(E):
        ref = wide.solve("cvar", b["idx_mpc"][e], b["init_state"][e], b["mean_param"][e], b["cov_param"][e], b["x_obs_traj"][e], b["y_obs_traj"][e],
                         b["v_des"][e])
        for k in _solve_keys("cvar"):
            _eq(got[k][e], ref[k], f"wide cvar {noise} episode {e} {k}")


# ---------------------------------------------------------------------------------------------------------------------------------
# the other instantiations: one small cell each

@gpu
@pytest.mark.parametrize("cell", list(OTHER_CELLS))
def test_instantiation_cell(mods, wl, sms, cell):
    kind, cost, nr, nobs, noise = OTHER_CELLS[cell]
    cem_impl, O = mods
    args = (nr, nobs, 0.3 if noise == "beta" else 0.1, 20 if nr > 5 else 30, noise, 0.05, 0.01)
    wide = nr > 64
    mk_ora = (lambda **kw: W.WideOracle(O, wl, nr, *args[1:], **kw)) if wide else (lambda **kw: O.OracleCEM(*args, **kw))
    if kind in ("stage", "fly_stage"):
        kw = INNER if cost == "mmd_opt" else {}
        n = _fly_samples(sms, nr) if kind == "fly_stage" else 6 if cost == "mmd_opt" else 12
        prob = cem_impl.CEM(*args, max_episodes=-(-n // 100), **kw); ora = mk_ora(**kw)
        rng = np.random.default_rng(len(cell))
        acc, steer = _controls(ora, rng, n)
        noise_t = ora.noise_tables(4242, 3)
        xo, yo, _ = ora.compute_obs_trajectories(*O.static_scene(nobs, 5))
        xo = np.ascontiguousarray(xo, f32); yo = np.ascontiguousarray(yo, f32)
        xo[0] = np.linspace(2, 60, 100); yo[0] = 1.75
        got = _launch(cell, lambda: prob.stage_risk(cost, acc, steer, ST0, noise_t, xo, yo))
        idx = range(n) if n <= 12 else sorted(set(range(0, n, 97)) | {n - 1})
        refs = _pool(lambda i: ora.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo), idx)
        _check(got, refs, _fields(cost), cell)
        assert np.any(got["risk"] != got["risk"][0]) or cost == "saa"
    else:
        E = _fly_episodes(sms, nr) if kind == "fly_solve" else 1
        kw = dict(maxiter_cem=2) if kind == "fly_solve" else SMALL if not wide else dict(num_batch=24, maxiter_cem=3)
        prob = cem_impl.CEM(*args, max_episodes=E, **kw); ora = mk_ora(**kw)
        b = _batch(O, ora, E, nobs)
        got = _launch(cell, lambda: prob.solve_batch(cost, **b))
        pick = range(E) if E <= 3 else sorted({0, E // 2, E - 1})
        refs = _pool(lambda e: _ref_solve(ora, cost, b, e), pick)
        for e, ref in refs.items():
            for k in _solve_keys(cost):
                _eq(got[k][e], ref[k], f"{cell} episode {e} {k}")
