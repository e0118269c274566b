"""Every supported num_reduced against the CPU oracle, bit for bit, at the shapes where the kernels branch.

mmd_opt takes num_reduced 2..40.  Above 10 its inner CEM is k_inner_cem_big, whose blocked Cholesky and resampling end in a partial panel
and super-panel that depend on d = num_reduced^2 + 1: d mod 16 is 1, 2, 5 or 10, which leaves one or two live columns in the last 4-column
panel and 4, 8 or 12 columns in the last 16-column super-panel.  The kernel has two launch shapes: 1024 threads when a launch has at most
one chain per SM, 256 otherwise; and its chain state lives in one fixed scratch, launched in turn as chain ranges when a launch holds more
chains than fit.  cvar, saa and mmd_random take num_reduced up to 64: their risk is ranked / summed by a warp in two halves (rollout
i = lane + 32 h), k_rollouts packs 128 / num_reduced samples into a CTA, and small launches stage the controls (ROLL_STAGED) while large
ones draw them on the fly (ROLL_FLY).  Each of these is run here on both sides of its boundary."""
import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
f32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
FIELDS = ("risk", "lane", "beta", "sigma", "res_beta")
ST0 = np.array([0.0, 1.75, 5.0, 0.0, 0.0], f32)
INNER = dict(num_samples_cem=40, maxiter_beta_cem=2)                 # reduced inner-CEM population: 40 samples, 5 elites, 2 iterations
SMALL = dict(num_batch=24, maxiter_cem=3, num_samples_cem=40, maxiter_beta_cem=4)
ROLL_THREADS = 128                                                    # k_rollouts CTA size (csrc/k_risk.cuh)
BIG_SCRATCH_BYTES = 8 << 30                                           # MPCMMD_BIG_SCRATCH_BYTES (csrc/mpcmmd_api.cu)


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


def _pair(mods, args, max_episodes=1, kernel="laplace", **kw):
    cem_impl, O = mods
    return cem_impl.CEM(*args, max_episodes=max_episodes, kernel=kernel, **kw), O.OracleCEM(*args, **kw)


def _episodes_for(n, num_batch=100):
    """max_episodes of a handle whose workspace (max_episodes * num_batch samples) holds a stage launch of n samples"""
    return -(-n // num_batch)


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
    return ((acc[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32), (steer[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32))


def _scene(O, ora, k=5, num_obs=2):
    xo, yo, _ = ora.compute_obs_trajectories(*O.static_scene(num_obs, k))
    xo = xo.copy(); xo[0] = np.linspace(2, 60, 100); yo = yo.copy(); yo[0] = 1.75      # an obstacle on the path: rollouts collide
    return xo, yo


def _oracle_risk(ora, cost, acc, steer, noise_t, xo, yo, idx):
    """ora.risk of the samples idx, one CPU thread per sample (the oracle's C entry keeps no global state, and ctypes releases the GIL)"""
    idx = [int(i) for i in idx]
    with ThreadPoolExecutor(max_workers=max(1, min(len(idx), os.cpu_count() or 1))) as ex:
        return dict(zip(idx, ex.map(lambda i: ora.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo), idx)))


def _check(got, refs, fields, what):
    for i, ref in refs.items():
        for k in fields:
            _eq(got[k][i], ref[k], f"{what} sample {i} {k}")


def _parts(prob, cost, acc, steer, noise_t, xo, yo, size):
    """the same stage as launches of at most `size` samples each, outputs concatenated"""
    outs = [prob.stage_risk(cost, acc[a:a + size], steer[a:a + size], ST0, noise_t, xo, yo) for a in range(0, len(acc), size)]
    return {k: np.concatenate([o[k] for o in outs]) for k in outs[0]}


# ---------------------------------------------------------------------------------------------------------------------------------
# mmd_opt at every num_reduced

def _d_mod16_row(nr):
    return (nr * nr + 1) % 16


@pytest.mark.parametrize("nr,noise", [(nr, "gaussian") for nr in range(2, 41)] + [(nr, "beta") for nr in (3, 7, 11, 14, 15, 16, 29, 40)])
def test_stage_risk_mmd_opt_every_num_reduced(mods, nr, noise):
    """three chains of mmd_opt's risk stage: k_inner_cem_lat (2..5 at this launch size), the generic k_inner_cem (6..10) and k_inner_cem_big
    (11..40) against the oracle, which is generic in num_reduced.  Above 10 this runs every tail of the blocked Cholesky: d mod 16 = 1, 2, 5
    and 10 (last panel with one or two live columns, last super-panel of 4, 8 or 12 columns) and every d mod 8 of the resampling."""
    cem_impl, O = mods
    prob, ora = _pair(mods, (nr, 2, 0.3 if noise == "beta" else 0.1, 20, noise, 0.05, 0.01), **INNER)
    acc, steer = _controls(ora, np.random.default_rng(1000 + nr), 3)
    noise_t = ora.noise_tables(4242, 3)
    xo, yo = _scene(O, ora)
    got = prob.stage_risk("mmd_opt", acc, steer, ST0, noise_t, xo, yo)
    _check(got, _oracle_risk(ora, "mmd_opt", acc, steer, noise_t, xo, yo, range(3)), FIELDS, f"mmd_opt nr={nr} {noise}")
    assert np.isfinite(got["res_beta"]).all()
    assert np.any(got["risk"] != f32(-1000.0)), "no chain collides: the risk does not depend on the reduced set"


def test_mmd_opt_sizes_cover_every_cholesky_tail():
    """the parametrisation above reaches each d mod 16 row of k_inner_cem_big with odd and even num_reduced"""
    rows = {}
    for nr in range(11, 41):
        rows.setdefault(_d_mod16_row(nr), set()).add(nr % 2)
    assert rows == {1: {0}, 5: {0}, 10: {1}, 2: {1}}


@pytest.fixture(scope="module")
def gk(mods, tmp_path_factory):
    """tests/gauss_oracle/oracle_gauss.c (the oracle with the MMD kernel form as a parameter) built with the oracle's flags into a temporary directory"""
    out = str(tmp_path_factory.mktemp("gauss_oracle") / "liboracle_gauss.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                           "-Wall", "-Wno-unused-function", "-Wno-misleading-indentation", "-Wno-maybe-uninitialized",
                           os.path.join(HERE, "gauss_oracle", "oracle_gauss.c"), "-o", out, "-lm"])
    lib = C.CDLL(out)
    lib.oracle_set_threads(min(32, os.cpu_count() or 1))
    return lib


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _gauss_risk(O, gk, ora, cost, acc, steer, noise_t, xo, yo):
    """OracleCEM.risk with the Gaussian MMD kernel (gk_risk of oracle_gauss.c, kernel form 1)"""
    z1, z2, z3, _, keys = noise_t
    nz = O.ONoise(_fp(z1), _fp(z2), _fp(z3), (C.c_uint32 * 2)(keys[0], keys[1]), (C.c_uint32 * 2)(keys[2], keys[3]), None, None)
    o = O.ORiskOut()
    acc = np.ascontiguousarray(acc, f32); steer = np.ascontiguousarray(steer, f32); st0 = np.ascontiguousarray(ST0, f32)
    xo = np.ascontiguousarray(xo, f32); yo = np.ascontiguousarray(yo, f32)
    gk.gk_risk(ora._cfg_for(cost), 1, O.COST_KINDS[cost], _fp(acc), _fp(steer), _fp(st0), C.byref(nz), _fp(xo), _fp(yo), C.byref(o))
    nr = ora.num_reduced
    return dict(risk=f32(o.risk), lane=f32(o.lane), beta=np.array(o.beta[:nr], f32), sigma=f32(o.sigma),
                res_beta=np.array(o.res_beta[:ora.iters_in], f32))


@pytest.mark.parametrize("nr", [11, 14, 15, 16])
def test_stage_risk_mmd_opt_gaussian_kernel_cholesky_tails(mods, gk, nr):
    """k_inner_cem_big with the Gaussian MMD kernel, one size from each d mod 16 row (10, 5, 2, 1), against the kernel-form oracle"""
    cem_impl, O = mods
    args = (nr, 2, 0.1, 20, "gaussian", 0.05, 0.01)
    prob, ora = _pair(mods, args, kernel="gaussian", **INNER)
    acc, steer = _controls(ora, np.random.default_rng(2000 + nr), 3)
    noise_t = ora.noise_tables(77, 1)
    xo, yo = _scene(O, ora)
    got = prob.stage_risk("mmd_opt", acc, steer, ST0, noise_t, xo, yo)
    lap = ora.risk("mmd_opt", acc[0], steer[0], ST0, noise_t, xo, yo)
    for i in range(3):
        ref = _gauss_risk(O, gk, ora, "mmd_opt", acc[i], steer[i], noise_t, xo, yo)
        for k in FIELDS:
            _eq(got[k][i], ref[k], f"gaussian nr={nr} chain {i} {k}")
    assert np.isfinite(got["res_beta"]).all()
    assert not np.array_equal(got["res_beta"][0], lap["res_beta"])           # the kernel form reached the device


# ---------------------------------------------------------------------------------------------------------------------------------
# k_inner_cem_big: launch shapes

@pytest.mark.parametrize("nr", [11, 13])
def test_inner_cem_big_256_thread_build(mods, sms, nr):
    """one launch of SMs + 1 chains takes the 256-thread build of k_inner_cem_big; every chain equals the same chain from launches of at most
    SMs chains (the 1024-thread build), and the first, the last and ten more equal the oracle"""
    cem_impl, O = mods
    n = sms + 1
    prob, ora = _pair(mods, (nr, 2, 0.1, 20, "gaussian", 0.05, 0.01), max_episodes=_episodes_for(n), **INNER)
    rng = np.random.default_rng(3000 + nr)
    acc, steer = _controls(ora, rng, n)
    noise_t = ora.noise_tables(57, 3)
    xo, yo = _scene(O, ora)
    got = prob.stage_risk("mmd_opt", acc, steer, ST0, noise_t, xo, yo)
    small = _parts(prob, "mmd_opt", acc, steer, noise_t, xo, yo, (n + 1) // 2)
    assert (n + 1) // 2 <= sms
    for k in FIELDS:
        _eq(got[k], small[k], f"nr={nr} {k}: {n} chains in one launch (256 threads) vs launches of <= {sms} (1024 threads)")
    pick = sorted({0, n - 1} | {int(i) for i in np.linspace(1, n - 2, 10)})
    _check(got, _oracle_risk(ora, "mmd_opt", acc, steer, noise_t, xo, yo, pick), FIELDS, f"nr={nr} 256 threads")
    assert len(np.unique(got["res_beta"][:, -1])) > n // 2                 # chains differ: a chain reading another's state would show


def _big_layout_floats(nr, S, ne):
    """floats per chain of k_inner_cem_big's state block: big_layout of csrc/k_inner_big.cuh, restated"""
    al4 = lambda x: (x + 3) & ~3
    nm = nr * nr; d = nm + 1; ldc = al4(d); kstride = al4(2 * nr * nr + 4 * nr)
    q = al4(nm * nm)                                                               # D
    q += al4(S * d) + al4(S) + al4(S * nr) + al4(S * nr)                           # th, cost, betas, idxs
    q += al4(S * nr) + al4(2 * S) + al4(S)                                         # rs, key64, perm
    q += d * ldc + al4(d)                                                          # C, mean
    q += al4(ne * d) + al4(ne * d) + al4(ne) + al4(ne * nr) + al4(ne * nr)          # eth, xc, ecost, ebetas, eidxs
    q += S * kstride + 256                                                         # kscr, small
    return (q + 31) & ~31


def test_big_layout_restatement_sizes():
    """the restated layout matches the per-chain sizes the kernel's documentation quotes (1.9 MB at nr 20, 23 MB at nr 40 with 100 samples)"""
    assert 1.8e6 < _big_layout_floats(20, 100, 11) * 4 < 2.0e6
    assert 22e6 < _big_layout_floats(40, 100, 11) * 4 < 23e6
    assert BIG_SCRATCH_BYTES // (_big_layout_floats(40, 100, 11) * 4) == 378
    assert BIG_SCRATCH_BYTES // (_big_layout_floats(40, 40, 5) * 4) == 401


def test_inner_cem_big_chain_ranges(mods, sms):
    """num_reduced 40: a launch of more chains than the 8 GiB chain scratch holds runs as successive chain ranges that reuse the same state
    blocks.  The handle allocates that full scratch.  n = one range + 9 chains; the chains around the range boundary and the last one equal
    the oracle, and every chain equals the same chain from launches of at most SMs chains (single range, 1024-thread build).  Two solves pin the
    library's range size to the restated r: one of r chains issues one k_inner_cem_big launch, one of r + 1 chains two."""
    cem_impl, O = mods
    nr = 40
    ne = max(int(0.1 * INNER["num_samples_cem"]) + 1, 3)
    r = BIG_SCRATCH_BYTES // (_big_layout_floats(nr, INNER["num_samples_cem"], ne) * 4)
    n = r + 9
    assert n > r > sms
    args = (nr, 2, 0.1, 20, "gaussian", 0.05, 0.01)
    prob, ora = _pair(mods, args, max_episodes=_episodes_for(n), maxiter_cem=1, **INNER)
    rng = np.random.default_rng(4000)
    acc, steer = _controls(ora, rng, n)
    noise_t = ora.noise_tables(4242, 3)
    xo, yo = _scene(O, ora)
    got = prob.stage_risk("mmd_opt", acc, steer, ST0, noise_t, xo, yo)
    small = _parts(prob, "mmd_opt", acc, steer, noise_t, xo, yo, sms)
    for k in FIELDS:
        _eq(got[k], small[k], f"{k}: {n} chains in ranges of {r} vs launches of <= {sms}")
    _check(got, _oracle_risk(ora, "mmd_opt", acc, steer, noise_t, xo, yo, [r - 2, r - 1, r, r + 1, n - 1]), FIELDS, f"nr=40 ranges of {r}")
    assert np.isfinite(got["res_beta"]).all()
    del prob                                                                       # each handle holds its own 8 GiB scratch
    # one outer iteration, one episode of num_batch chains: the launch counts differ only by the number of chain ranges
    from mpcmmd_b200 import scenes
    counts = []
    for B in (r, r + 1):
        p = cem_impl.CEM(*args, max_episodes=1, num_batch=B, maxiter_cem=1, **INNER)
        p.solve_batch("mmd_opt", **scenes.static_batch(p, [0]))
        counts.append(p.last_launch_count())
        del p
    assert counts[1] == counts[0] + 1, (r, counts)


# ---------------------------------------------------------------------------------------------------------------------------------
# cvar, saa, mmd_random: num_reduced rollouts per sample

def _roll_spb(nr, num_prime, n, sms):
    """samples per CTA of k_rollouts for cvar / saa / mmd_random: roll_spb of csrc/mpcmmd_api.cu with roll_smem_floats of csrc/k_risk.cuh, restated"""
    stage = n * nr < 2 * sms * ROLL_THREADS                                        # roll_stage_ctrl
    tail = 16 if nr <= 16 else (nr + 3) & ~3
    smem_bytes = lambda spb: 4 * spb * (4 * tail + (2 * nr * num_prime if stage else 0))
    spb = max(1, ROLL_THREADS // nr)
    if stage:
        spb = min(spb, 8)
    while spb > 1 and smem_bytes(spb) > 96 * 1024:
        spb -= 1
    while spb > 1 and -(-n // spb) < 4 * sms:
        spb -= 1
    return min(spb, 2) if stage else spb


@pytest.mark.parametrize("side", ["staged", "fly"])
@pytest.mark.parametrize("nr", [2, 3, 31, 32, 33, 47, 63, 64])
@pytest.mark.parametrize("cost", ["cvar", "saa", "mmd_random"])
def test_stage_risk_num_reduced_rollout_costs(mods, sms, cost, nr, side):
    """the warp-parallel risk of num_reduced rollouts (ranks and kernel rows of i = lane and lane + 32: 31 / 32 / 33 straddle the halves, 64 fills
    both) on both sides of the switch between staged controls (5 samples, one per CTA) and controls drawn on the fly (n * nr >= 2 * SMs * 128).
    The large launch has enough samples that k_rollouts packs the most its CTA holds, 128 // num_reduced samples (64 at nr 2, 42 at 3, 4 at 31 / 32,
    3 at 33, 2 at 47 / 63 / 64); the restated roll_spb asserts it.  Odd sizes 3, 33, 63 run beta noise.  Every sample of the small launch and a strided subset
    plus the last sample of the large one equal the oracle."""
    cem_impl, O = mods
    thr = 2 * sms * ROLL_THREADS
    n = 5 if side == "staged" else max(-(-thr // nr) + 7, 4 * sms * (ROLL_THREADS // nr) + 7)
    assert (n * nr < thr) == (side == "staged")
    assert _roll_spb(nr, 20, n, sms) == (1 if side == "staged" else ROLL_THREADS // nr)
    noise = "beta" if nr in (3, 33, 63) else "gaussian"
    prob, ora = _pair(mods, (nr, 2, 0.3 if noise == "beta" else 0.1, 20, noise, 0.05, 0.01), max_episodes=_episodes_for(n))
    acc, steer = _controls(ora, np.random.default_rng(5000 + nr), n)
    noise_t = ora.noise_tables(91, 2)
    xo, yo = _scene(O, ora)
    got = prob.stage_risk(cost, acc, steer, ST0, noise_t, xo, yo)
    idx = range(n) if side == "staged" else sorted(set(range(0, n, max(1, n // 48))) | {n - 1})
    fields = ("risk", "lane", "beta", "sigma") if cost == "mmd_random" else ("risk", "lane")
    _check(got, _oracle_risk(ora, cost, acc, steer, noise_t, xo, yo, idx), fields, f"{cost} nr={nr} {noise} {side} n={n}")
    assert np.isfinite(got["risk"]).all()
    if cost != "saa":
        assert np.any(got["risk"] != got["risk"][0])


# ---------------------------------------------------------------------------------------------------------------------------------
# full solves above num_reduced 5

def _solve_inputs(O, ora, E):
    eps = [O.static_episode(2, k) for k in range(E)]
    tr = [ora.compute_obs_trajectories(*sc) for sc, _ in eps]
    return [i for _, i in eps], np.stack([t[0] for t in tr]), np.stack([t[1] for t in tr])


@pytest.mark.parametrize("cost,nr,noise,E", [("mmd_opt", 8, "gaussian", 3), ("mmd_opt", 13, "gaussian", 3), ("cvar", 33, "beta", 3),
                                             ("cvar", 64, "gaussian", 2)])
def test_solve_large_num_reduced_bit_exact(mods, cost, nr, noise, E):
    """the solve graph at num_reduced 8 (generic inner kernel), 13 (k_inner_cem_big, odd) and 33 / 64 (cvar): write_rolls, the episode views of
    the stored mother rollouts and the num_reduced-long beta records k_select copies out, against OracleCEM.solve"""
    cem_impl, O = mods
    prob, ora = _pair(mods, (nr, 2, 0.3 if noise == "beta" else 0.1, 30, noise, 0.02, 0.01), max_episodes=E, **SMALL)
    init_state, mean, cov, v_des = O.driver_inputs("static")
    idx, xo, yo = _solve_inputs(O, ora, E)
    got = prob.solve_batch(cost, idx, np.stack([init_state] * E), np.stack([mean] * E), np.stack([cov] * E), xo, yo, [v_des] * E)
    for e in range(E):
        ref = ora.solve(cost, idx[e], init_state, mean, cov, xo[e], yo[e], v_des)
        for k in ("cx", "cy", "cost_obs", "cost_lane") + (("beta", "sigma", "res_beta") if cost == "mmd_opt" else ()):
            _eq(got[k][e], ref[k], f"{cost} nr={nr} ep{e} {k}")
    assert np.isfinite(got["cx"]).all()


def test_grouped_solve_graph_large_num_reduced(mods, monkeypatch):
    """MPCMMD_GROUPS=2 at num_reduced 12: k_inner_cem_big keeps its chains in one scratch shared by every episode, so the solve stays one group
    (two branches would run the kernel concurrently on the same chain blocks).  Every episode equals the same episode solved alone and the
    oracle, and the grouped handle issues the launches of one group."""
    cem_impl, O = mods
    from mpcmmd_b200 import scenes
    E = 3
    args = (12, 2, 0.1, 30, "gaussian", 0.02, 0.01)
    monkeypatch.setenv("MPCMMD_GROUPS", "2")
    big = cem_impl.CEM(*args, max_episodes=E, **SMALL)
    monkeypatch.delenv("MPCMMD_GROUPS")
    one = cem_impl.CEM(*args, max_episodes=1, **SMALL)
    ora = O.OracleCEM(*args, **SMALL)
    batch = scenes.static_batch(big, list(range(E)))
    out = big.solve_batch("mmd_opt", **batch)
    grouped_launches = big.last_launch_count()
    for k in range(E):
        solo = one.solve_batch("mmd_opt", **{n: v[k:k + 1] for n, v in batch.items()})
        ref = ora.solve("mmd_opt", int(batch["idx_mpc"][k]), batch["init_state"][k], batch["mean_param"][k], batch["cov_param"][k],
                        batch["x_obs_traj"][k], batch["y_obs_traj"][k], float(batch["v_des"][k]))
        for f in ("cx", "cy", "cost_obs", "cost_lane", "beta", "sigma", "res_beta"):
            _eq(out[f][k], solo[f][0], f"episode {k} {f}: MPCMMD_GROUPS=2 vs alone")
            _eq(out[f][k], ref[f], f"episode {k} {f}: MPCMMD_GROUPS=2 vs oracle")
    assert grouped_launches == one.last_launch_count()


def test_inner_cem_path_names_the_kernel(mods):
    cem_impl, _ = mods
    for nr, want in ((5, "k_inner_cem_fast "), (8, "k_inner_cem (generic"), (13, "k_inner_cem_big ")):
        prob = cem_impl.CEM(nr, 2, 0.1, 20, "gaussian", 0.0, 0.0, max_episodes=1, num_batch=24)
        assert prob.inner_cem_path().startswith(want), (nr, prob.inner_cem_path())
