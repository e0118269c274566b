"""Gaussian-kernel MMD (opt-in, `kernel="gaussian"`; DESIGN.md section 3 item 8): the kernel entry, an independent float64 restatement of
the reduced-set inner CEM and of the scalar-cost MMD with that kernel, the driver / validation tags, and on the GPU the device paths
(fast, latency, generic and large-reduced-set inner-CEM kernels, k_opt_risk, mmd_random's warp MMD) against the oracle bit for bit.
Laplace stays the default; a default run is unchanged.

The CPU reference with the kernel form as a parameter is tests/gauss_oracle/oracle_gauss.c: the frozen oracle (oracle/) compiled into the
same unit, with its inner CEM, scalar MMD, risk stage and solve restated for either form.  Its Laplace form is checked bit for bit against
the frozen oracle here, which pins the restatement to it."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

f32 = np.float32
FIELDS = ("risk", "lane", "beta", "sigma", "res_beta")


HERE = os.path.dirname(os.path.abspath(__file__))
KERNELS = {"laplace": 0, "gaussian": 1}


@pytest.fixture(scope="module")
def O(built):
    from oracle import oracle
    return oracle


@pytest.fixture(scope="module")
def gk(O, tmp_path_factory):
    """tests/gauss_oracle/oracle_gauss.c built with the oracle's flags into a temporary directory"""
    out = str(tmp_path_factory.mktemp("gauss_oracle") / "liboracle_gauss.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                           "-Wall", "-Wno-unused-function", "-Wno-misleading-indentation", "-Wno-maybe-uninitialized",
                           os.path.join(HERE, "gauss_oracle", "oracle_gauss.c"), "-o", out, "-lm"])
    lib = C.CDLL(out)
    lib.oracle_set_threads(min(32, os.cpu_count() or 1))
    return lib


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def entry(gk, kernel, q, sigma):
    """the inner-CEM kernel entry k(q; sigma) of the form"""
    q = np.ascontiguousarray(q, f32); sigma = np.ascontiguousarray(sigma, f32); out = np.empty_like(q)
    gk.gk_entry_vec(KERNELS[kernel], _fp(q), _fp(sigma), _fp(out), int(q.size))
    return out


class KernelOracle:
    """OracleCEM (constants, configuration, projection, noise tables) whose risk stage and solve take the MMD kernel form: the same
    call surface as OracleCEM.risk / .solve, computed by oracle_gauss.c"""

    def __init__(self, O, gk, *args, kernel="laplace", **kw):
        self._O, self._gk, self.kernel = O, gk, kernel
        self._ora = O.OracleCEM(*args, **kw)

    def __getattr__(self, name):
        return getattr(self._ora, name)

    def risk(self, cost, acc, steer, st0, noise, x_obs_traj, y_obs_traj, want_rollouts=False, beta_draws=None):
        O, ora = self._O, self._ora
        z1, z2, z3, _, keys = noise
        b1 = b2 = None
        if beta_draws is not None:
            b1, b2 = (np.ascontiguousarray(b, f32).reshape(-1) for b in beta_draws)
        nz = O.ONoise(_fp(z1), _fp(z2), _fp(z3), (C.c_uint32 * 2)(keys[0], keys[1]), (C.c_uint32 * 2)(keys[2], keys[3]),
                      _fp(b1) if b1 is not None else None, _fp(b2) if b2 is not None else None)
        o = O.ORiskOut()
        acc = np.ascontiguousarray(acc, f32); steer = np.ascontiguousarray(steer, f32); st0 = np.ascontiguousarray(st0, f32)
        xo = np.ascontiguousarray(x_obs_traj, f32); yo = np.ascontiguousarray(y_obs_traj, f32)
        self._gk.gk_risk(ora._cfg_for(cost), KERNELS[self.kernel], O.COST_KINDS[cost], _fp(acc), _fp(steer), _fp(st0), C.byref(nz),
                         _fp(xo), _fp(yo), C.byref(o))
        nr = self.num_reduced
        d = dict(risk=f32(o.risk), lane=f32(o.lane), beta=np.array(o.beta[:nr], f32), sigma=f32(o.sigma),
                 res_beta=np.array(o.res_beta[:self.iters_in], f32), red_cost=np.array(o.red_cost[:nr], f32),
                 red_idx=np.array(o.red_idx[:nr], np.int32))
        if want_rollouts:              # the rollouts do not depend on the kernel: the frozen oracle's
            r = ora.risk(cost, acc, steer, st0, noise, xo, yo, want_rollouts=True, beta_draws=beta_draws)
            d["x_roll"], d["y_roll"] = r["x_roll"], r["y_roll"]
        return d

    def solve(self, cost, idx_mpc, init_state, mean, cov, x_obs_traj, y_obs_traj, v_des):
        O, ora = self._O, self._ora
        init_state = np.ascontiguousarray(init_state, f32); mean = np.ascontiguousarray(mean, f32)
        cov = np.ascontiguousarray(cov, f32); xo = np.ascontiguousarray(x_obs_traj, f32); yo = np.ascontiguousarray(y_obs_traj, f32)
        out = O.OSolveOut()
        self._gk.gk_solve(ora._cfg_for(cost), KERNELS[self.kernel], O.COST_KINDS[cost], C.c_int32(int(idx_mpc)), _fp(init_state), _fp(mean),
                          _fp(cov), _fp(xo), _fp(yo), C.c_float(v_des), C.byref(out))
        nr = self.num_reduced
        return dict(cx=np.array(out.cx, f32), cy=np.array(out.cy, f32), cost_lane=f32(out.cost_lane), cost_obs=f32(out.cost_obs),
                    beta=np.array(out.beta[:nr], f32), sigma=f32(out.sigma), res_beta=np.array(out.res_beta[:self.iters_in], f32),
                    sel=int(out.sel_last))


def _eq(a, b, what):
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if not np.array_equal(a, b, equal_nan=True):
        bad = np.flatnonzero(~((a == b) | (np.isnan(a) & np.isnan(b))).ravel())
        raise AssertionError(f"{what}: {bad.size}/{a.size} elements differ; first at {bad[:5]}: got {a.ravel()[bad[:5]]} want {b.ravel()[bad[:5]]}")


def _controls(ora, rng, n):
    beq_x = np.array([0.0, 5.0, 0.0], f32); beq_y = np.array([1.75, 0.0, 0.0, 0.0], f32)
    acc, steer = [], []
    for _ in range(n):
        p = np.concatenate([rng.uniform(2, 25, 4), rng.normal(0, 3, 4)]).astype(f32)
        o = ora.project(p, beq_x, beq_y, 15.0, np.zeros(11, f32), np.zeros(11, f32), np.zeros(198, f32))
        acc.append(o["acc"]); steer.append(o["steer"])
    return np.stack(acc), np.stack(steer)


def _scene(O, ora, k=3, num_obs=2):
    xo, yo, _ = ora.compute_obs_trajectories(*O.static_scene(num_obs, k))
    xo = xo.copy(); xo[0] = np.linspace(2, 60, 100); yo = yo.copy(); yo[0] = 1.75      # an obstacle on the path: nonzero costs
    return xo, yo


ST0 = np.array([0.0, 1.75, 5.0, 0.0, 0.0], f32)


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: the entry

def test_gaussian_entry_special_values(gk):
    """k(0) = 1 exactly; NaN distance or bandwidth gives NaN; q beyond the cap 125 / g2 gives the capped value 2^-125 (also for q = inf)"""
    sig = np.array([0.01, 0.5, 1.0, 7.0, 1e3], f32)
    _eq(entry(gk, "gaussian", np.zeros(5, f32), sig), np.ones(5, f32), "k(0)")
    assert np.isnan(entry(gk, "gaussian", np.array([np.nan, 1.0], f32), np.array([1.0, np.nan], f32))).all()
    for s in (0.01, 1.0, 3.0):
        g2 = f32(f32(f32(1.0) / f32(s)) ** 2) * f32(0.72134752044448170)
        cap = f32(125.0) / g2
        q = np.array([cap, cap * f32(2), np.float32(np.inf), f32(1e30)], f32)
        k = entry(gk, "gaussian", q, np.full(4, s, f32))
        assert (k == k[0]).all() and k[0] > 0 and abs(float(k[0]) / 2.0 ** -125 - 1.0) < 125 * math.log(2) * 2.0 ** -23, (s, k)      # dcap * g2 = 125 (1 + 2^-24 at most)


def test_gaussian_entry_accuracy(gk):
    """|k / exp(-q / (2 sigma^2)) - 1| <= 5e-6 for q / (2 sigma^2) <= 16, with q and sigma the float32 arguments.
    Derivation: g2 = RN(RN(RN(1/sigma)^2) * RN(log2 e) / 2) carries five roundings (the reciprocal enters squared), so
    g2 = g2* (1 + d) with |d| <= 5u, u = 2^-24.  The entry is 2^(-q g2), hence its relative error from d is ln 2 * q g2* |d| = (q / (2 sigma^2)) |d|
    <= 16 * 5u = 4.77e-6.  The reduced argument f takes one rounding (|f| <= 1/2: 2^-25 absolute, 2.1e-8 relative), P6 approximates 2^f to 3.9e-9
    and its Horner evaluation and the final product add at most 2u = 1.2e-7: 4.77e-6 + 2.1e-8 + 3.9e-9 + 1.2e-7 < 5e-6."""
    rng = np.random.default_rng(11)
    n = 400000
    sig = np.exp(rng.uniform(np.log(0.01), np.log(20.0), n)).astype(f32)
    x = rng.uniform(0.0, 16.0, n)
    q = (x * 2.0 * sig.astype(np.float64) ** 2).astype(f32)
    ex = np.exp(-q.astype(np.float64) / (2.0 * sig.astype(np.float64) ** 2))
    keep = q.astype(np.float64) / (2.0 * sig.astype(np.float64) ** 2) <= 16.0
    k = entry(gk, "gaussian", q, sig).astype(np.float64)
    err = np.abs(k[keep] / ex[keep] - 1.0)
    assert err.max() <= 5e-6, err.max()
    assert err.max() > 1e-7          # the bound is not vacuous: the scale's roundings show at large arguments


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: independent float64 restatement (DESIGN.md Appendix D.5 with the Gaussian kernel)

def _gauss(q, s):
    return np.exp(-q / (2.0 * s * s))


def _inner_iteration_f64(ora, F, theta):
    """one inner iteration of compute_beta on every row of theta: top-nr |theta|, K_mix, K_red, the (nr + 1) KKT system and the cost"""
    nr, nm = ora.num_reduced, ora.num_mother
    D = ((F[:, None, :] - F[None, :, :]) ** 2).sum(-1)                       # squared L2 distances of the 22 features
    costs, betas, idxs = [], [], []
    for row in theta.astype(np.float64):
        idx = np.argsort(np.abs(row[:nm]), kind="stable")[nm - nr:]
        s = row[nm]
        Kmix = _gauss(D[idx], s)                                             # (nr, nm)
        Kred = _gauss(D[np.ix_(idx, idx)], s)
        A = np.zeros((nr + 1, nr + 1)); A[:nr, :nr] = Kred + 0.05 * np.eye(nr); A[:nr, nr] = 1.0; A[nr, :nr] = 1.0
        rhs = np.concatenate([Kmix.sum(1) / nm, [1.0]])
        beta = np.linalg.solve(A, rhs)[:nr]
        costs.append(beta @ Kred @ beta - 2.0 / nm * Kmix.sum(1) @ beta)
        betas.append(beta); idxs.append(idx)
    return np.array(costs), betas, idxs


@pytest.mark.parametrize("nr", [2, 5, 10])
def test_inner_cem_restatement(O, gk, nr):
    """teacher-forced on the oracle's mother rollouts and theta0: the best cost, its reduced set and its weights of one inner iteration"""
    ora = KernelOracle(O, gk, nr, 2, 0.1, 20, "gaussian", 0.0, 0.0, num_samples_cem=40, maxiter_beta_cem=1, kernel="gaussian")
    acc, steer = _controls(ora, np.random.default_rng(3 + nr), 1)
    noise_t = ora.noise_tables(17, 0)
    xo, yo = _scene(O, ora)
    ref = ora.risk("mmd_opt", acc[0], steer[0], ST0, noise_t, xo, yo, want_rollouts=True)
    W = ora.Wfit.astype(np.float64)
    F = np.concatenate([ref["x_roll"].astype(np.float64) @ W.T, ref["y_roll"].astype(np.float64) @ W.T], 1)
    costs, betas, idxs = _inner_iteration_f64(ora, F, ora.theta0)
    best = int(np.argmin(costs))
    scale = max(1.0, float(np.abs(costs).max()))
    assert abs(costs[best] - float(ref["res_beta"][0])) <= 1e-4 * scale, (costs[best], ref["res_beta"][0])
    np.testing.assert_array_equal(idxs[best], ref["red_idx"])
    np.testing.assert_allclose(ref["beta"], betas[best], rtol=1e-4, atol=1e-4)


def _mmd_f64(c, beta, sigma, nr, ker_wt=1000.0):
    c = np.asarray(c, np.float64); beta = np.asarray(beta, np.float64)
    K = _gauss((c[:, None] - c[None, :]) ** 2, float(sigma))
    k0 = _gauss(c ** 2, float(sigma))
    return ker_wt * (beta @ K @ beta - 2.0 * (beta @ k0))


@pytest.mark.parametrize("cost", ["mmd_opt", "mmd_random"])
def test_scalar_cost_mmd_restatement(O, gk, cost):
    """the risk value of the chosen reduced set (kernel_computation.py:67-87 with the Gaussian kernel); mmd_random: beta = 1/nr, sigma = 0.01"""
    nr = 5
    ora = KernelOracle(O, gk, nr, 2, 0.1, 20, "gaussian", 0.0, 0.0, num_samples_cem=40, maxiter_beta_cem=3, kernel="gaussian")
    acc, steer = _controls(ora, np.random.default_rng(8), 4)
    noise_t = ora.noise_tables(5, 1)
    xo, yo = _scene(O, ora)
    seen = 0
    for i in range(4):
        ref = ora.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo)
        if cost == "mmd_random":
            assert ref["sigma"] == f32(0.01) and np.all(ref["beta"] == f32(1.0 / nr))
        want = _mmd_f64(ref["red_cost"], ref["beta"], ref["sigma"], nr)
        assert abs(float(ref["risk"]) - want) <= 1e-4 * max(1.0, abs(want)), (i, ref["risk"], want)
        seen += np.any(ref["red_cost"] > 0)
    assert seen                       # at least one sample sees the obstacle


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: the kernel-form oracle's Laplace form is the frozen oracle, and the kernel choice is validated

@pytest.mark.parametrize("cost", ["mmd_opt", "mmd_random", "cvar"])
@pytest.mark.parametrize("noise,naive", [("gaussian", False), ("beta", False), ("gaussian", True)])
def test_kernel_oracle_laplace_is_the_oracle(O, gk, cost, noise, naive):
    """bit for bit on full solves and on the risk stage (the naive path recomputes the distances per beta sample)"""
    kw = dict(num_batch=24, maxiter_cem=2, num_samples_cem=40, maxiter_beta_cem=3, naive=naive)
    args = (5, 2, 0.3 if noise == "beta" else 0.1, 30, noise, 0.02, 0.01)
    ref, lap, gau = O.OracleCEM(*args, **kw), KernelOracle(O, gk, *args, **kw), KernelOracle(O, gk, *args, kernel="gaussian", **kw)
    init_state, mean, cov, v_des = O.driver_inputs("static")
    (sc, idx) = O.static_episode(2, 1)
    xo, yo, _ = ref.compute_obs_trajectories(*sc)
    ra, rl, rg = (o.solve(cost, idx, init_state, mean, cov, xo, yo, v_des) for o in (ref, lap, gau))
    for k in ("cx", "cy", "cost_obs", "cost_lane", "beta", "sigma", "res_beta", "sel"):
        _eq(rl[k], ra[k], k)
    xo, yo = _scene(O, ref)
    acc, steer = _controls(ref, np.random.default_rng(4), 3)
    noise_t = ref.noise_tables(11, 1)
    for i in range(3):
        a, l = ref.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo), lap.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo)
        for k in FIELDS + ("red_cost", "red_idx"):
            _eq(l[k], a[k], f"risk[{i}] {k}")
    if cost == "mmd_opt":             # the form reaches the restatement
        assert not np.array_equal(rg["res_beta"], ra["res_beta"])


def test_unknown_kernel_refused(built):
    from mpcmmd_b200 import cem_impl
    with pytest.raises(ValueError):
        cem_impl.CEM(5, 2, 0.1, 30, "gaussian", 0.0, 0.0, kernel="cauchy")


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: driver and validation files

@pytest.fixture(scope="module")
def driver(built):
    from mpcmmd_b200 import driver
    return driver


def _fake_out(episodes):
    E = len(episodes)
    return dict(cost_obs=np.full(E, -1500.0, f32), cost_lane=np.zeros(E, f32), cx=np.ones((E, 11), f32), cy=np.ones((E, 11), f32))


class _FakeCEM:
    ker_wt = 1000.0
    made = []

    def __init__(self, *a, kernel="laplace", **kw):
        self.kernel = kernel
        _FakeCEM.made.append(kernel)

    def solve_batch(self, cost, episodes):
        return _fake_out(episodes)


def _sweep(driver, monkeypatch, tmp_path, extra):
    monkeypatch.setattr(driver, "CEM", _FakeCEM)
    monkeypatch.setattr(driver.scenes, "static_batch", lambda prob, mine, variant: dict(episodes=mine))
    args = driver.build_parser().parse_args(["--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "2", "--costs", "mmd_opt",
                                             "mmd_random", "cvar", "saa", "--num_prime", "30", "--noises", "beta", "--acc_const_noise", "0",
                                             "--steer_const_noise", "0", "--num_configs", "4", "--root", str(tmp_path)] + extra)
    files = driver.run_sweep(args, log=lambda *a: None)
    return args, {c: dict(np.load(p)) for p in files for c in ("mmd_opt", "mmd_random", "cvar", "saa") if os.path.basename(p).startswith(c + "_")}


def test_driver_kernel_flag(driver, monkeypatch, tmp_path):
    p = driver.build_parser()
    base = ["--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "2", "--costs", "mmd_opt", "--num_prime", "30", "--noises", "beta",
            "--acc_const_noise", "0", "--steer_const_noise", "0"]
    assert p.parse_args(base).kernel == "laplace"
    assert p.parse_args(base + ["--kernel", "gaussian"]).kernel == "gaussian"
    with pytest.raises(SystemExit):
        p.parse_args(base + ["--kernel", "cauchy"])
    _, default = _sweep(driver, monkeypatch, tmp_path / "a", [])
    keys = {"cx", "cy", "init_state", "x_obs", "y_obs", "vx_obs", "vy_obs"}
    assert set(default) == {"mmd_opt", "mmd_random", "cvar", "saa"}
    for name, d in default.items():
        assert set(d) == keys, name
    _FakeCEM.made.clear()
    _, gauss = _sweep(driver, monkeypatch, tmp_path / "b", ["--kernel", "gaussian"])
    assert _FakeCEM.made == ["gaussian"]
    for name, d in gauss.items():
        if name.startswith("mmd"):
            assert set(d) == keys | {"kernel"} and str(d["kernel"]) == "gaussian", name
        else:
            assert set(d) == keys, name
            for k in keys:
                np.testing.assert_array_equal(d[k], default[name][k])


def test_validation_stats_inherit_kernel(driver, monkeypatch, tmp_path):
    from mpcmmd_b200 import validation as V
    for extra, want in (([], None), (["--kernel", "gaussian"], "gaussian")):
        root = tmp_path / ("g" if want else "l")
        args, _ = _sweep(driver, monkeypatch, root / "data", extra)
        monkeypatch.setattr(V, "CEM", _FakeCEM)
        monkeypatch.setattr(V, "compute_stats_batch", lambda prob, items, *a, **k: (np.zeros(len(items), np.int32), np.zeros(len(items), np.int32)))
        vargs = V.build_parser().parse_args(["--noise_levels", "0.3", "--num_reduced_sets", "5", "--num_obs", "2", "--num_prime", "30",
                                             "--noises", "beta", "--acc_const_noise", "0", "--steer_const_noise", "0",
                                             "--root", str(root / "data"), "--stats_root", str(root / "stats")])
        (path,) = V.run_validation(vargs, log=lambda *a: None)
        st = np.load(path)
        if want is None:
            assert "kernel" not in st.files
        else:
            assert str(st["kernel"]) == want


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU

@pytest.fixture(scope="module")
def mods(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mpcmmd_b200 import cem_impl
    from oracle import oracle
    oracle.set_threads(min(32, os.cpu_count() or 1))
    return cem_impl, oracle


@pytest.fixture(scope="module")
def KO(mods, gk):
    """KernelOracle with the frozen oracle module and the kernel-form library bound"""
    return lambda *a, **kw: KernelOracle(mods[1], gk, *a, **kw)


@pytest.mark.gpu
def test_device_gaussian_entry_bit_exact(mods, gk):
    """math_vec fn 13 (dm::lap_ with dm::kern_scale<KER_GAUSSIAN>) == the oracle, including capped, zero, infinite and NaN arguments"""
    cem_impl, O = mods
    rng = np.random.default_rng(7)
    q = np.concatenate([rng.uniform(0, 60, 300000), rng.uniform(0, 1e6, 199993), [0.0, -0.0, np.inf, np.nan, 1.0, 1.0, 3.0]]).astype(f32)
    sig = np.concatenate([rng.uniform(0.01, 4.0, 499993), [1.0, 1.0, 0.01, 1.0, np.nan, np.inf, 0.0]]).astype(f32)
    assert q.size == 500000
    _eq(cem_impl.math_vec(13, q, sig), entry(gk, "gaussian", q, sig), "gauss")


def _stage(mods, KO, monkeypatch, cost, nr, noise, kw, n=3, mode=None, seed=1):
    cem_impl, O = mods
    if mode:
        monkeypatch.setenv("MPCMMD_INNER_CEM", mode)
    args = (nr, 2, 0.3 if noise == "beta" else 0.1, 20, noise, 0.02, 0.01)
    prob = cem_impl.CEM(*args, max_episodes=1, kernel="gaussian", **kw)
    ora = KO(*args, kernel="gaussian", **kw)
    acc, steer = _controls(ora, np.random.default_rng(seed + nr), n)
    noise_t = ora.noise_tables(77, 1)
    xo, yo = _scene(O, ora)
    got = prob.stage_risk(cost, acc, steer, ST0, noise_t, xo, yo)
    for i in range(n):
        ref = ora.risk(cost, acc[i], steer[i], ST0, noise_t, xo, yo)
        for k in (FIELDS if cost == "mmd_opt" else ("risk", "lane")):
            _eq(got[k][i], ref[k], f"{cost} nr={nr} {noise} chain {i} {k}")
    return prob, got


SMALL_IN = dict(num_samples_cem=40, maxiter_beta_cem=4)


@pytest.mark.gpu
@pytest.mark.parametrize("noise", ["gaussian", "beta"])
@pytest.mark.parametrize("nr,mode,kw", [(2, "cta", SMALL_IN), (3, None, SMALL_IN), (5, "cta", dict(maxiter_beta_cem=3)), (5, "lat", SMALL_IN),
                                        (5, None, dict(maxiter_beta_cem=3)), (6, None, SMALL_IN), (8, None, SMALL_IN), (10, None, dict(maxiter_beta_cem=2)),
                                        (12, None, dict(num_samples_cem=30, maxiter_beta_cem=2)), (20, None, dict(num_samples_cem=30, maxiter_beta_cem=2))])
def test_stage_risk_mmd_opt_gaussian(mods, KO, monkeypatch, noise, nr, mode, kw):
    """k_inner_cem_fast (cta: throughput build; lat: its latency build), k_inner_cem_lat (default at this launch size, nr <= 5), the generic
    k_inner_cem (nr 6..10; nr = 10 at the reference's population: the 100 / 11 build) and k_inner_cem_big (nr 12, 20)"""
    prob, got = _stage(mods, KO, monkeypatch, "mmd_opt", nr, noise, kw, mode=mode)
    assert np.isfinite(got["res_beta"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("noise", ["gaussian", "beta"])
def test_stage_risk_mmd_random_gaussian(mods, KO, monkeypatch, noise):
    _, got = _stage(mods, KO, monkeypatch, "mmd_random", 5, noise, {}, n=6)
    assert np.isfinite(got["risk"]).all()


@pytest.mark.gpu
def test_stage_risk_injected_gaussian(mods, KO):
    cem_impl, O = mods
    nr, npr = 5, 30
    args = (nr, 3, 0.3, npr, "beta", 0.05, 0.01)
    prob = cem_impl.CEM(*args, max_episodes=1, kernel="gaussian", **SMALL_IN)
    ora = KO(*args, kernel="gaussian", **SMALL_IN)
    rng = np.random.default_rng(29)
    n = 4
    acc, steer = _controls(ora, rng, n)
    noise_t = ora.noise_tables(99, 1)
    xo, yo = _scene(O, ora, 4, 3)
    b_acc = np.stack([rng.beta(2 * np.maximum(np.abs(acc[i][:npr]), 1e-3), 5 * np.maximum(np.abs(acc[i][:npr]), 1e-3), (nr, npr)) for i in range(n)]).astype(f32)
    b_steer = np.stack([rng.beta(2 * np.maximum(np.abs(steer[i][:npr]), 1e-3), 5 * np.maximum(np.abs(steer[i][:npr]), 1e-3), (nr, npr)) for i in range(n)]).astype(f32)
    got = prob.stage_risk_injected("mmd_opt", acc, steer, ST0, noise_t[2], b_acc, b_steer, xo, yo)
    for i in range(n):
        ref = ora.risk("mmd_opt", acc[i], steer[i], ST0, noise_t, xo, yo, beta_draws=(b_acc[i], b_steer[i]))
        for k in FIELDS:
            _eq(got[k][i], ref[k], f"{k}[{i}]")


def _solve_check(prob, ora, O, cost, E, num_obs=2):
    init_state, mean, cov, v_des = O.driver_inputs("static")
    eps = [O.static_episode(num_obs, k) for k in range(E)]
    tr = [ora.compute_obs_trajectories(*sc) for sc, _ in eps]
    idx, xo, yo = [i for _, i in eps], np.stack([t[0] for t in tr]), np.stack([t[1] for t in tr])
    got = prob.solve_batch(cost, idx, np.stack([init_state] * E), np.stack([mean] * E), np.stack([cov] * E), xo, yo, [v_des] * E)
    for e in range(E):
        ref = ora.solve(cost, idx[e], init_state, mean, cov, xo[e], yo[e], v_des)
        for k in ("cx", "cy", "cost_obs", "cost_lane") + (("beta", "sigma", "res_beta") if cost == "mmd_opt" else ()):
            _eq(got[k][e], ref[k], f"{cost} ep{e} {k}")
    return got


@pytest.mark.gpu
@pytest.mark.parametrize("cost", ["mmd_opt", "mmd_random"])
@pytest.mark.parametrize("E", [1, 5])
def test_solve_gaussian_bit_exact(mods, KO, cost, E):
    """one episode (100 chains: the latency builds) and five (500 chains > 3 per SM: the throughput kernel)"""
    cem_impl, O = mods
    kw = dict(num_batch=100, maxiter_cem=2, num_samples_cem=40, maxiter_beta_cem=3)
    args = (5, 2, 0.1, 30, "gaussian", 0.02, 0.01)
    prob = cem_impl.CEM(*args, max_episodes=E, kernel="gaussian", **kw)
    _solve_check(prob, KO(*args, kernel="gaussian", **kw), O, cost, E)


@pytest.mark.gpu
def test_handles_keep_their_kernel(mods, KO):
    """a Laplace and a Gaussian handle of one configuration, used alternately, each give their own kernel's results; a handle from
    mpcmmd_create equals one from mpcmmd_create_with_kernel(LAPLACE) bit for bit"""
    cem_impl, O = mods
    kw = dict(num_batch=24, maxiter_cem=2, num_samples_cem=40, maxiter_beta_cem=3)
    args = (5, 2, 0.1, 30, "gaussian", 0.02, 0.01)
    lap, gau = cem_impl.CEM(*args, max_episodes=2, **kw), cem_impl.CEM(*args, max_episodes=2, kernel="gaussian", **kw)
    assert lap.kernel == "laplace" and gau.kernel == "gaussian"
    olap, ogau = O.OracleCEM(*args, **kw), KO(*args, kernel="gaussian", **kw)
    outs = []
    for _ in range(2):
        outs.append(_solve_check(lap, olap, O, "mmd_opt", 2))
        outs.append(_solve_check(gau, ogau, O, "mmd_opt", 2))
    assert not np.array_equal(outs[0]["res_beta"], outs[1]["res_beta"])
    plain = cem_impl.CEM(*args, max_episodes=2, **kw)
    from mpcmmd_b200 import binding as B
    h = C.c_void_p()
    B.check(plain._lib.mpcmmd_create(C.byref(plain._cfg), 0, C.byref(h)))
    plain._lib.mpcmmd_destroy(plain._h)
    plain._h = h
    got = _solve_check(plain, olap, O, "mmd_opt", 2)
    for k in ("cx", "cy", "cost_obs", "cost_lane", "beta", "sigma", "res_beta"):
        _eq(got[k], outs[0][k], k)


@pytest.mark.gpu
def test_unknown_kernel_refused_by_abi(mods):
    cem_impl, _ = mods
    prob = cem_impl.CEM(5, 2, 0.1, 30, "gaussian", 0.0, 0.0, max_episodes=1, num_batch=24)
    h = C.c_void_p()
    assert prob._lib.mpcmmd_create_with_kernel(C.byref(prob._cfg), 2, 0, C.byref(h)) != 0
    assert b"mmd_kernel" in prob._lib.mpcmmd_last_error()


@pytest.mark.gpu
def test_fast_math_gaussian_within_tolerance(mods, KO, monkeypatch):
    """MPCMMD_MATH=fast with a Gaussian handle: the exponentials on MUFU.EX2, held at the fast-math test's 1e-4 (beta at 20x) against the exact
    Gaussian oracle"""
    cem_impl, O = mods
    monkeypatch.setenv("MPCMMD_MATH", "fast")
    monkeypatch.setenv("MPCMMD_INNER_CEM", "cta")
    args = (5, 2, 0.1, 20, "gaussian", 0.0, 0.0)
    kw = dict(maxiter_beta_cem=3)
    prob = cem_impl.CEM(*args, max_episodes=1, kernel="gaussian", **kw)
    ora = KO(*args, kernel="gaussian", **kw)
    acc, steer = _controls(ora, np.random.default_rng(12), 3)
    noise_t = ora.noise_tables(40, 1)
    xo, yo = _scene(O, ora)
    got = prob.stage_risk("mmd_opt", acc, steer, ST0, noise_t, xo, yo)
    for i in range(3):
        ref = ora.risk("mmd_opt", acc[i], steer[i], ST0, noise_t, xo, yo)
        np.testing.assert_allclose(got["res_beta"][i], ref["res_beta"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(got["sigma"][i], ref["sigma"], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(got["risk"][i], ref["risk"], rtol=1e-4, atol=1e-4 * 1000)
        np.testing.assert_allclose(got["beta"][i], ref["beta"], rtol=2e-3, atol=2e-3)


@pytest.mark.gpu
@pytest.mark.parametrize("var,val", [("MPCMMD_INNER_CEM", "warp"), ("MPCMMD_INNER_CEM", "pipe"), ("MPCMMD_INNER_CEM", "split"),
                                     ("MPCMMD_CHOL", "la"), ("MPCMMD_CHOL", "cta")])
def test_experimental_variants_refuse_gaussian(mods, monkeypatch, var, val):
    cem_impl, _ = mods
    from mpcmmd_b200 import binding as B
    monkeypatch.setenv(var, val)
    with pytest.raises(B.MpcmmdError, match="Laplace only"):
        cem_impl.CEM(5, 2, 0.1, 30, "gaussian", 0.0, 0.0, max_episodes=1, num_batch=24, kernel="gaussian")
