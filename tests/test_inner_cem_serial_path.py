"""The one-warp phases of the reduced-set inner CEM (k_inner_cem_fast) against the CPU oracle, bit for bit, on the inputs that take their
less common branches:

* the panel Cholesky's last panel, which has fewer than four live columns whenever d = nr^2 + 1 is not a multiple of four
  (nr = 2, 3, 4, 5: d = 5, 10, 17, 26, i.e. one or two live columns),
* the selection on tied costs: with noise-free rollouts every mother rollout is the same, the distance table is all zeros and a sample's
  cost depends on its bandwidth alone, so every sample whose bandwidth was clipped to the floor ties with every other such sample;
  a NaN control makes every cost NaN (all keys tie at "NaN last"),
* iteration 0 at the reference's population (100 samples on 96 threads: four threads evaluate a second sample).

The CTA-per-chain kernel is forced (MPCMMD_INNER_CEM=cta): a launch this small would otherwise take a latency build, which factors in
registers instead."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
f32 = np.float32
FIELDS = ("risk", "lane", "beta", "sigma", "res_beta")


@pytest.fixture(scope="module")
def mods(built):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from mpcmmd_b200 import cem_impl
    from oracle import oracle as O
    return cem_impl, O


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


def _run(mods, monkeypatch, nr, noise_level, kw, n=4, seed=5, poison=None):
    """n chains of the mmd_opt risk stage through k_inner_cem_fast and through the oracle; poison(acc, steer) may edit the controls"""
    cem_impl, O = mods
    monkeypatch.setenv("MPCMMD_INNER_CEM", "cta")
    args = (nr, 2, noise_level, 20, "gaussian", 0.0, 0.0)
    prob = cem_impl.CEM(*args, variant="static", max_episodes=1, **kw)
    ora = O.OracleCEM(*args, variant="static", **kw)
    acc, steer = _controls(ora, np.random.default_rng(seed + nr), n)
    if poison is not None:
        poison(acc, steer)
    st0 = np.array([0.0, 1.75, 5.0, 0.0, 0.0], f32)
    noise_t = ora.noise_tables(321, 1)
    xo, yo, _ = ora.compute_obs_trajectories(*O.static_scene(2, 3))
    xo = xo.copy(); xo[0] = np.linspace(2, 60, 100); yo = yo.copy(); yo[0] = 1.75
    got = prob.stage_risk("mmd_opt", acc, steer, st0, noise_t, xo, yo)
    refs = [ora.risk("mmd_opt", acc[i], steer[i], st0, noise_t, xo, yo) for i in range(n)]
    for i, ref in enumerate(refs):
        for k in FIELDS:
            _eq(got[k][i], ref[k], f"nr={nr} chain {i} {k}")
    return got, refs


@pytest.mark.parametrize("nr", [2, 3, 4, 5])
def test_partial_last_panel_reference_population(mods, monkeypatch, nr):
    """reference population (100 samples, 11 elites; nr = 5 runs the build with those sizes as template constants), 5 iterations"""
    got, _ = _run(mods, monkeypatch, nr, 0.1, dict(maxiter_beta_cem=5))
    assert np.isfinite(got["res_beta"]).all()


@pytest.mark.parametrize("nr", [3, 5])
def test_tied_costs_from_noise_free_rollouts(mods, monkeypatch, nr):
    """noise level 0: all costs of samples with the floored bandwidth are equal; the stable order (lowest candidate index first) decides"""
    got, refs = _run(mods, monkeypatch, nr, 0.0, dict(maxiter_beta_cem=4))
    # the premise: the best cost of every iteration is shared by several candidates, so ties were actually resolved
    ora_th = mods[1].OracleCEM(nr, 2, 0.0, 20, "gaussian", 0.0, 0.0, variant="static").theta0
    assert (ora_th[:, -1] == f32(0.01)).sum() > 11
    assert np.isfinite(got["res_beta"]).all()


def test_nan_costs_keep_the_stable_order(mods, monkeypatch):
    """a NaN control turns every mother rollout, every distance and so every sample cost of that chain into NaN: all keys tie"""
    def poison(acc, steer):
        acc[1, 7] = np.nan
    got, refs = _run(mods, monkeypatch, 5, 0.1, dict(maxiter_beta_cem=3), poison=poison)
    assert np.isnan(refs[1]["res_beta"]).all() and np.isfinite(got["res_beta"][0]).all()
