"""Every instantiation of the reduced-set inner CEM of mmd_opt against the oracle, each cell checked by the name of the kernel it launched.

launch_risk (csrc/mpcmmd_api.cu) picks the inner-CEM kernel from five things: num_reduced, the inner population (num_samples_cem S and
from it num_ellite_beta ne = max(int(0.1 S) + 1, 3)), the MMD kernel form (KER 0 Laplace, 1 Gaussian), MPCMMD_MATH=fast, and the launch's
chain count.  The k_inner_cem_fast family serves num_reduced <= 5 with S <= 128 and ne <= 12: at most SMs chains run k_inner_cem_lat (16
warps per chain), at most 3 SMs chains the latency build k_inner_cem_fast<LAT>, larger launches its throughput build (or, with
MPCMMD_MATH=fast, the fast-math build FM, tolerance parity only).  Everything else runs the generic k_inner_cem (num_reduced <= 10) or
k_inner_cem_big (1024 threads for at most SMs chains, 256 above).  The reference's population (S = 100, ne = 11) has builds with those sizes
as template constants (SC / NEC).  MPCMMD_INNER_CEM=cta|lat|lat512|generic, read at create, forces a family member whatever the launch size.

Templates: k_inner_cem_fast<NR, LAT, FM, SC, NEC, KER>, k_inner_cem_lat<NR, SC, NEC, KER>, k_inner_cem<NR, SC, NEC, KER>,
k_inner_cem_big<THREADS, KER>.

The populations reach the fast kernels' less common branches: S - ne > 96 resampled rows (a second pass of the 96-thread resampling loop,
and the latency build's unrolled path instead of its prefetched normals), ne = 3, 4, 10 (divisors of the covariance other than the
reference's 10), ne = 12 (the most elites the gather and covariance take), S < 32 (lanes of the one-warp selection without a candidate) and
S = 4 (one resampled row).  S = 120 (ne = 13) and S > 128 leave the fast family.  Within one population every exact build gives the same
bits for the same chain; Laplace cells equal OracleCEM, Gaussian cells the kernel-form oracle tests/gauss_oracle/oracle_gauss.c."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import kernel_names as KN

gpu = pytest.mark.gpu
f32 = np.float32
ST0 = np.array([0.0, 1.75, 5.0, 0.0, 0.0], f32)
FIELDS = ("risk", "lane", "beta", "sigma", "res_beta")
SOLVE_KEYS = ("cx", "cy", "cost_obs", "cost_lane", "beta", "sigma", "res_beta")
ICF_THREADS, ICF_MAX_S, ICF_MAX_NE = 96, 128, 12                       # csrc/k_inner_cem.cuh
MAX_S = 8 * 96                                                         # RISKO_THREADS * 8: the largest population create accepts
MODES = ("cta", "lat", "lat512", "generic")

# ---------------------------------------------------------------------------------------------------------------------------------
# cells

POPS = (4, 31, 33, 97, 107, 108, 110, 119)
# (kernel form, num_reduced, S): nr 5 Laplace at every population and at the reference's (the SC / NEC = 100 / 11 builds); nr 2..4 Laplace
# and nr 2..5 Gaussian on a subset, each at a small and a large population
POP_CASES = ([("laplace", 5, S) for S in POPS + (100,)]
             + [("laplace", 2, 4), ("laplace", 2, 97), ("laplace", 3, 31), ("laplace", 3, 110), ("laplace", 4, 33), ("laplace", 4, 108)]
             + [("gaussian", 2, 4), ("gaussian", 2, 119), ("gaussian", 3, 33), ("gaussian", 3, 107), ("gaussian", 4, 31), ("gaussian", 4, 110),
                ("gaussian", 5, 108), ("gaussian", 5, 119), ("gaussian", 5, 100)])
# populations the fast family does not take (ne 13 at S = 120, S > 128): the generic kernel whatever MPCMMD_INNER_CEM asks for
SWITCH_CASES = [("laplace", 120, "auto"), ("laplace", 120, "cta"), ("gaussian", 120, "lat512"), ("laplace", 257, "lat"),
                ("gaussian", 257, "auto"), ("laplace", MAX_S, "auto"), ("gaussian", MAX_S, "cta")]
# num_reduced 6..10: the generic kernel at the reference's population (the 100 / 11 builds) and at run-time sizes; lat512 / cta overrides
# above num_reduced 5 fall back to it
REF_CASES = ([(ker, nr, S, "auto") for ker in ("laplace", "gaussian") for nr in range(6, 11) for S in (100, 40)]
             + [("laplace", 8, 100, "lat512"), ("gaussian", 7, 33, "cta")])
AUTO_POINTS = ("sm", "sm+1", "3sm", "3sm+1")
AUTO_S = {"laplace": 40, "gaussian": 110}
FM_CASES = [(ker, nr, S) for ker in ("laplace", "gaussian") for nr, S in ((2, 40), (3, 40), (4, 40), (5, 40), (5, 100))]
SOLVE_CASES = {
    # cell: (kernel form, num_reduced, S, maxiter_beta_cem, num_batch: an int or a multiple of the SM count) -- two episodes each
    "solve/laplace/S119": ("laplace", 5, 119, 3, "2sm"),       # 4 SMs chains: throughput build
    "solve/laplace/S4": ("laplace", 5, 4, 3, 24),              # 48 chains: k_inner_cem_lat
    "solve/laplace/iters1": ("laplace", 5, 40, 1, "sm"),       # 2 SMs chains: latency build
    "solve/laplace/iters64": ("laplace", 5, 40, 64, 24),
    "solve/gaussian/S33": ("gaussian", 5, 33, 3, 24),
}


def _pop(ker, nr, mode, ref=False):
    """population cells of (ker, nr) forced to `mode`, at the reference's population or at the others"""
    cells = [f"pop/{k}/{n}/{S}/{mode}" for k, n, S in POP_CASES if k == ker and n == nr and (S == 100) == ref]
    return cells + ([f"pop0/laplace/5/119/{mode}"] if (ker, nr, ref) == ("laplace", 5, False) else [])


def _ref(ker, nr, ref):
    return [f"ref/{k}/{n}/{S}/{m}" for k, n, S, m in REF_CASES if k == ker and n == nr and (S == 100) == ref]


def _switch(ker):
    return [f"switch/{k}/{S}/{m}" for k, S, m in SWITCH_CASES if k == ker]


def _fm(ker, nr, ref=False):
    return [f"fm/{k}/{n}/{S}" for k, n, S in FM_CASES if k == ker and n == nr and (S == 100) == ref]


# instantiation -> the cells below that launch it (each launch asserts that exactly the instantiations listed for it ran)
TABLE = {
    "k_inner_cem_fast<2, false, false, 0, 0, 0>": _pop("laplace", 2, "cta"),
    "k_inner_cem_fast<3, false, false, 0, 0, 0>": _pop("laplace", 3, "cta"),
    "k_inner_cem_fast<4, false, false, 0, 0, 0>": _pop("laplace", 4, "cta"),
    "k_inner_cem_fast<5, false, false, 0, 0, 0>": _pop("laplace", 5, "cta") + ["auto/laplace/3sm+1", "solve/laplace/S119"],
    "k_inner_cem_fast<5, false, false, 100, 11, 0>": _pop("laplace", 5, "cta", ref=True),
    "k_inner_cem_fast<2, true, false, 0, 0, 0>": _pop("laplace", 2, "lat"),
    "k_inner_cem_fast<3, true, false, 0, 0, 0>": _pop("laplace", 3, "lat"),
    "k_inner_cem_fast<4, true, false, 0, 0, 0>": _pop("laplace", 4, "lat"),
    "k_inner_cem_fast<5, true, false, 0, 0, 0>": _pop("laplace", 5, "lat") + ["auto/laplace/sm+1", "auto/laplace/3sm", "auto_fm/laplace/3sm",
                                                                             "solve/laplace/iters1"],
    "k_inner_cem_fast<5, true, false, 100, 11, 0>": _pop("laplace", 5, "lat", ref=True),
    "k_inner_cem_fast<2, false, true, 0, 0, 0>": _fm("laplace", 2),
    "k_inner_cem_fast<3, false, true, 0, 0, 0>": _fm("laplace", 3),
    "k_inner_cem_fast<4, false, true, 0, 0, 0>": _fm("laplace", 4),
    "k_inner_cem_fast<5, false, true, 0, 0, 0>": _fm("laplace", 5) + ["auto_fm/laplace/3sm+1"],
    "k_inner_cem_fast<5, false, true, 100, 11, 0>": _fm("laplace", 5, ref=True),
    "k_inner_cem_fast<2, false, false, 0, 0, 1>": _pop("gaussian", 2, "cta"),
    "k_inner_cem_fast<3, false, false, 0, 0, 1>": _pop("gaussian", 3, "cta"),
    "k_inner_cem_fast<4, false, false, 0, 0, 1>": _pop("gaussian", 4, "cta"),
    "k_inner_cem_fast<5, false, false, 0, 0, 1>": _pop("gaussian", 5, "cta") + ["auto/gaussian/3sm+1"],
    "k_inner_cem_fast<5, false, false, 100, 11, 1>": _pop("gaussian", 5, "cta", ref=True),
    "k_inner_cem_fast<2, true, false, 0, 0, 1>": _pop("gaussian", 2, "lat"),
    "k_inner_cem_fast<3, true, false, 0, 0, 1>": _pop("gaussian", 3, "lat"),
    "k_inner_cem_fast<4, true, false, 0, 0, 1>": _pop("gaussian", 4, "lat"),
    "k_inner_cem_fast<5, true, false, 0, 0, 1>": _pop("gaussian", 5, "lat") + ["auto/gaussian/sm+1", "auto/gaussian/3sm", "auto_fm/gaussian/3sm"],
    "k_inner_cem_fast<5, true, false, 100, 11, 1>": _pop("gaussian", 5, "lat", ref=True),
    "k_inner_cem_fast<2, false, true, 0, 0, 1>": _fm("gaussian", 2),
    "k_inner_cem_fast<3, false, true, 0, 0, 1>": _fm("gaussian", 3),
    "k_inner_cem_fast<4, false, true, 0, 0, 1>": _fm("gaussian", 4),
    "k_inner_cem_fast<5, false, true, 0, 0, 1>": _fm("gaussian", 5) + ["auto_fm/gaussian/3sm+1"],
    "k_inner_cem_fast<5, false, true, 100, 11, 1>": _fm("gaussian", 5, ref=True),
    "k_inner_cem_lat<2, 0, 0, 0>": _pop("laplace", 2, "lat512"),
    "k_inner_cem_lat<3, 0, 0, 0>": _pop("laplace", 3, "lat512"),
    "k_inner_cem_lat<4, 0, 0, 0>": _pop("laplace", 4, "lat512"),
    "k_inner_cem_lat<5, 0, 0, 0>": _pop("laplace", 5, "lat512") + ["auto/laplace/sm", "auto/laplace/parts", "solve/laplace/S4",
                                                                  "solve/laplace/iters64"],
    "k_inner_cem_lat<5, 100, 11, 0>": _pop("laplace", 5, "lat512", ref=True),
    "k_inner_cem_lat<2, 0, 0, 1>": _pop("gaussian", 2, "lat512"),
    "k_inner_cem_lat<3, 0, 0, 1>": _pop("gaussian", 3, "lat512"),
    "k_inner_cem_lat<4, 0, 0, 1>": _pop("gaussian", 4, "lat512"),
    "k_inner_cem_lat<5, 0, 0, 1>": _pop("gaussian", 5, "lat512") + ["auto/gaussian/sm", "auto/gaussian/parts", "solve/gaussian/S33"],
    "k_inner_cem_lat<5, 100, 11, 1>": _pop("gaussian", 5, "lat512", ref=True),
    "k_inner_cem<2, 0, 0, 0>": _pop("laplace", 2, "generic"),
    "k_inner_cem<3, 0, 0, 0>": _pop("laplace", 3, "generic"),
    "k_inner_cem<4, 0, 0, 0>": _pop("laplace", 4, "generic"),
    "k_inner_cem<5, 0, 0, 0>": _pop("laplace", 5, "generic") + _pop("laplace", 5, "generic", ref=True) + _switch("laplace"),
    "k_inner_cem<6, 0, 0, 0>": _ref("laplace", 6, False),
    "k_inner_cem<7, 0, 0, 0>": _ref("laplace", 7, False),
    "k_inner_cem<8, 0, 0, 0>": _ref("laplace", 8, False),
    "k_inner_cem<9, 0, 0, 0>": _ref("laplace", 9, False),
    "k_inner_cem<10, 0, 0, 0>": _ref("laplace", 10, False),
    "k_inner_cem<6, 100, 11, 0>": _ref("laplace", 6, True),
    "k_inner_cem<7, 100, 11, 0>": _ref("laplace", 7, True),
    "k_inner_cem<8, 100, 11, 0>": _ref("laplace", 8, True),
    "k_inner_cem<9, 100, 11, 0>": _ref("laplace", 9, True),
    "k_inner_cem<10, 100, 11, 0>": _ref("laplace", 10, True),
    "k_inner_cem<2, 0, 0, 1>": _pop("gaussian", 2, "generic"),
    "k_inner_cem<3, 0, 0, 1>": _pop("gaussian", 3, "generic"),
    "k_inner_cem<4, 0, 0, 1>": _pop("gaussian", 4, "generic"),
    "k_inner_cem<5, 0, 0, 1>": _pop("gaussian", 5, "generic") + _pop("gaussian", 5, "generic", ref=True) + _switch("gaussian"),
    "k_inner_cem<6, 0, 0, 1>": _ref("gaussian", 6, False),
    "k_inner_cem<7, 0, 0, 1>": _ref("gaussian", 7, False),
    "k_inner_cem<8, 0, 0, 1>": _ref("gaussian", 8, False),
    "k_inner_cem<9, 0, 0, 1>": _ref("gaussian", 9, False),
    "k_inner_cem<10, 0, 0, 1>": _ref("gaussian", 10, False),
    "k_inner_cem<6, 100, 11, 1>": _ref("gaussian", 6, True),
    "k_inner_cem<7, 100, 11, 1>": _ref("gaussian", 7, True),
    "k_inner_cem<8, 100, 11, 1>": _ref("gaussian", 8, True),
    "k_inner_cem<9, 100, 11, 1>": _ref("gaussian", 9, True),
    "k_inner_cem<10, 100, 11, 1>": _ref("gaussian", 10, True),
    "k_inner_cem_big<1024, 0>": ["big/laplace/sm"],
    "k_inner_cem_big<256, 0>": ["big/laplace/sm+1"],
    "k_inner_cem_big<1024, 1>": ["big/gaussian/sm"],
    "k_inner_cem_big<256, 1>": ["big/gaussian/sm+1"],
}


def _cell_keys():
    keys = {f"pop/{k}/{n}/{S}/{m}" for k, n, S in POP_CASES for m in MODES} | {f"pop0/laplace/5/119/{m}" for m in MODES}
    keys |= {f"switch/{k}/{S}/{m}" for k, S, m in SWITCH_CASES}
    keys |= {f"ref/{k}/{n}/{S}/{m}" for k, n, S, m in REF_CASES}
    keys |= {f"auto/{k}/{p}" for k in AUTO_S for p in AUTO_POINTS + ("parts",)} | {f"auto_fm/{k}/{p}" for k in AUTO_S for p in ("3sm", "3sm+1")}
    keys |= {f"big/{k}/{p}" for k in AUTO_S for p in ("sm", "sm+1")}
    keys |= {f"fm/{k}/{n}/{S}" for k, n, S in FM_CASES}
    return keys | set(SOLVE_CASES)


def _want(cell):
    return {k for k, cells in TABLE.items() if cell in cells}


def _launch(cell, fn):
    """fn() under the profiler; asserts that the inner-CEM instantiations it ran are exactly those TABLE assigns to `cell`"""
    out, names = KN.launched(fn)
    ran = KN.family(names, "inner")
    assert ran == _want(cell), f"{cell}: expected {sorted(_want(cell))} to run, the profiler saw {sorted(ran)} (all kernels: {sorted(names)})"
    return out


def _is_fast(nr, S, ne):
    """inner_cem_is_fast of csrc/mpcmmd_api.cu, restated"""
    return nr <= 5 and S <= ICF_MAX_S and 2 <= ne <= ICF_MAX_NE and S - ne >= 1


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: the table covers exactly the instantiations the library holds; the populations reach the branches they are chosen for

def test_instantiation_table_matches_library(built):
    """the inner-CEM instantiations in libmpcmmd.so are exactly TABLE's keys, every cell TABLE names is one of this module's cells and every
    cell of this module is named, and no instantiation is left without a cell"""
    have = KN.built_instantiations(built.LIB, "inner")
    assert len(have) == 72, sorted(have)
    assert have == set(TABLE), f"in the library but not in TABLE: {sorted(have - set(TABLE))}; in TABLE but not built: {sorted(set(TABLE) - have)}"
    named = {c for cells in TABLE.values() for c in cells}
    assert named == _cell_keys(), (sorted(named - _cell_keys()), sorted(_cell_keys() - named))
    assert all(TABLE.values()), [k for k, v in TABLE.items() if not v]
    assert len(KN.built_instantiations(built.LIB)) == 25                 # the rollout family's view is unchanged


def test_populations_reach_the_branches(built):
    """the oracle's elite counts of the populations: every divisor branch of the covariance, the largest elite count the fast kernels take,
    both sides of one resampling pass (S - ne = 96 and 97+), selections with fewer than 32 candidates, a single resampled row, and the
    switch to the generic kernel at S = 120 and above 128.  The GPU cells hold each handle's num_ellite_beta to the oracle's."""
    from oracle import oracle as O
    ne = {S: O.OracleCEM(5, 2, 0.1, 20, "gaussian", 0.0, 0.0, num_samples_cem=S, maxiter_beta_cem=1).n_el_in for S in POPS + (100, 120, 257)}
    assert [ne[S] for S in POPS] == [3, 4, 4, 10, 11, 11, 12, 12]
    assert all(_is_fast(5, S, ne[S]) for S in POPS + (100,)) and not _is_fast(5, 120, ne[120]) and not _is_fast(5, 257, ne[257])
    rows = {S: S - ne[S] for S in POPS}
    assert rows[4] == 1 and rows[107] == ICF_THREADS and min(rows[S] for S in (108, 110, 119)) > ICF_THREADS
    assert {S for S in POPS if S < 32} == {4, 31} and ICF_MAX_NE in ne.values()
    assert {n for _, n, _ in POP_CASES} == {2, 3, 4, 5} and {S for k, n, S in POP_CASES if (k, n) == ("laplace", 5)} == set(POPS) | {100}


# ---------------------------------------------------------------------------------------------------------------------------------
# helpers

def _eq(a, b, what=""):
    a = np.asarray(a); b = np.asarray(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    if not np.array_equal(a, b, equal_nan=True):
        bad = np.flatnonzero(~((a == b) | (np.isnan(a) & np.isnan(b))).ravel())
        raise AssertionError(f"{what}: {bad.size}/{a.size} elements differ; first at {bad[:5]}: got {a.ravel()[bad[:5]]} want {b.ravel()[bad[:5]]}")


def _close(got, ref, what):
    """fast-math tolerance (the bounds of test_fast_math_gaussian_within_tolerance): res_beta and sigma 1e-4 relative and absolute, risk and
    lane 1e-4 relative and 0.1 absolute, beta 2e-3"""
    for k, rtol, atol in (("res_beta", 1e-4, 1e-4), ("sigma", 1e-4, 1e-4), ("risk", 1e-4, 0.1), ("lane", 1e-4, 0.1), ("beta", 2e-3, 2e-3)):
        np.testing.assert_allclose(got[k], ref[k], rtol=rtol, atol=atol, err_msg=f"{what} {k}")


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


def _args(nr, noise_level=0.1):
    return (nr, 2, noise_level, 20, "gaussian", 0.05 if noise_level else 0.0, 0.01 if noise_level else 0.0)


def _oracle(mods, gk, ker, args, **kw):
    """OracleCEM for the Laplace form, the kernel-form oracle for the Gaussian one"""
    from test_mmd_gaussian_kernel import KernelOracle
    _, O = mods
    return O.OracleCEM(*args, **kw) if ker == "laplace" else KernelOracle(O, gk, *args, kernel=ker, **kw)


def _handle(mods, monkeypatch, ker, args, n, mode="auto", fast_math=False, **kw):
    """a handle whose workspace holds a stage of n chains; MPCMMD_INNER_CEM and MPCMMD_MATH are read at create"""
    cem_impl, _ = mods
    monkeypatch.setenv("MPCMMD_INNER_CEM", mode)
    if fast_math:
        monkeypatch.setenv("MPCMMD_MATH", "fast")
    else:
        monkeypatch.delenv("MPCMMD_MATH", raising=False)
    prob = cem_impl.CEM(*args, max_episodes=-(-n // 100), kernel=ker, **kw)
    monkeypatch.delenv("MPCMMD_INNER_CEM")
    monkeypatch.delenv("MPCMMD_MATH", raising=False)
    return prob


def _controls(ora, rng, n, bases=12):
    """n control sequences: `bases` projected ones, each further sample a randomly scaled copy of one of them"""
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
    pick[:bases] = np.arange(bases)
    return ((acc[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32), (steer[pick] * rng.uniform(0.5, 1.5, (n, 1))).astype(f32))


def _inputs(mods, ora, n, seed):
    """controls of n chains, noise tables and a scene with an obstacle on the path (so the risk depends on the reduced set)"""
    _, O = mods
    acc, steer = _controls(ora, np.random.default_rng(seed), n)
    xo, yo, _ = ora.compute_obs_trajectories(*O.static_scene(2, 5))
    xo = np.ascontiguousarray(xo, f32); yo = np.ascontiguousarray(yo, f32)
    xo[0] = np.linspace(2, 60, 100); yo[0] = 1.75
    return dict(acc=acc, steer=steer, noise=ora.noise_tables(seed, 1), xo=xo, yo=yo)


def _stage(prob, inp, a=0, b=None):
    return prob.stage_risk("mmd_opt", inp["acc"][a:b], inp["steer"][a:b], ST0, inp["noise"], inp["xo"], inp["yo"])


def _parts(prob, inp, n, size):
    outs = [_stage(prob, inp, a, min(a + size, n)) for a in range(0, n, size)]
    return {k: np.concatenate([o[k] for o in outs]) for k in outs[0]}


def _refs(ora, inp, idx):
    """ora.risk of the chains idx, one CPU thread per chain"""
    idx = [int(i) for i in idx]
    fn = lambda i: ora.risk("mmd_opt", inp["acc"][i], inp["steer"][i], ST0, inp["noise"], inp["xo"], inp["yo"])
    with ThreadPoolExecutor(max_workers=max(1, min(len(idx), os.cpu_count() or 1))) as ex:
        return dict(zip(idx, ex.map(fn, idx)))


def _check(got, refs, what):
    for i, ref in refs.items():
        for k in FIELDS:
            _eq(got[k][i], ref[k], f"{what} chain {i} {k}")


def _same(a, b, what):
    for k in FIELDS:
        _eq(a[k], b[k], f"{what} {k}")


def _strided(n, marks, k=12):
    return sorted({int(i) for i in np.linspace(0, n - 1, k)} | {m for m in marks if 0 <= m < n})


# ---------------------------------------------------------------------------------------------------------------------------------
# populations through every exact fast-family build and the generic kernel

def _population(mods, gk, monkeypatch, ker, nr, S, noise_level, cell, n=8, iters=5, seed=0):
    ora = _oracle(mods, gk, ker, _args(nr, noise_level), num_samples_cem=S, maxiter_beta_cem=iters)
    ne = ora.n_el_in
    inp = _inputs(mods, ora, n, 100 * nr + S + seed)
    outs = {}
    for mode in MODES:
        prob = _handle(mods, monkeypatch, ker, _args(nr, noise_level), n, mode, num_samples_cem=S, maxiter_beta_cem=iters)
        assert prob.num_ellite_beta == ne and _is_fast(nr, S, ne)
        outs[mode] = _launch(f"{cell}/{mode}", lambda: _stage(prob, inp))
        del prob
    for mode in MODES[1:]:
        _same(outs[mode], outs["cta"], f"{cell}: {mode} vs cta, every chain")
    _check(outs["cta"], _refs(ora, inp, range(n)), cell)
    assert np.isfinite(outs["cta"]["res_beta"]).all()
    return outs["cta"], ora


@gpu
@pytest.mark.parametrize("ker,nr,S", POP_CASES)
def test_population(mods, gk, monkeypatch, ker, nr, S):
    """eight chains, five inner iterations, through k_inner_cem_fast (cta), its latency build (lat), k_inner_cem_lat (lat512) and the generic
    k_inner_cem: identical bits across the four, and equal to the oracle"""
    got, _ = _population(mods, gk, monkeypatch, ker, nr, S, 0.1, f"pop/{ker}/{nr}/{S}")
    assert len(np.unique(got["res_beta"][:, -1])) > 1 and np.any(got["risk"] != got["risk"][0])


@gpu
def test_population_noise_free_ties(mods, gk, monkeypatch):
    """noise level 0 at S = 119: every mother rollout is the same, so every sample whose bandwidth sits at the floor ties with every other
    such sample, and candidates 96 and up (the fourth slot of each lane of the one-warp selection) take part in the ties"""
    got, ora = _population(mods, gk, monkeypatch, "laplace", 5, 119, 0.0, "pop0/laplace/5/119")
    floor = np.flatnonzero(ora.theta0[:, -1] == f32(0.01))
    assert floor.size > ora.n_el_in and floor.max() >= ICF_THREADS


# ---------------------------------------------------------------------------------------------------------------------------------
# outside the fast family: the generic kernel

@gpu
@pytest.mark.parametrize("ker,S,mode", SWITCH_CASES)
def test_population_leaves_fast_family(mods, gk, monkeypatch, ker, S, mode):
    """S = 120 (13 elites), 257 and 768 (the largest population create accepts: 8 samples per thread of the 96-thread generic kernel): the
    generic kernel runs whatever MPCMMD_INNER_CEM asks for, and the handle reports it"""
    n, iters = 4, 2 if S == MAX_S else 3
    prob = _handle(mods, monkeypatch, ker, _args(5), n, mode, num_samples_cem=S, maxiter_beta_cem=iters)
    assert not _is_fast(5, S, prob.num_ellite_beta)
    assert prob.inner_cem_path().startswith("k_inner_cem (generic"), prob.inner_cem_path()
    ora = _oracle(mods, gk, ker, _args(5), num_samples_cem=S, maxiter_beta_cem=iters)
    assert ora.n_el_in == prob.num_ellite_beta
    inp = _inputs(mods, ora, n, S)
    got = _launch(f"switch/{ker}/{S}/{mode}", lambda: _stage(prob, inp))
    _check(got, _refs(ora, inp, range(n)), f"S={S} {ker} {mode}")


@gpu
def test_population_above_limit_refused(mods, monkeypatch):
    from mpcmmd_b200 import binding as B
    with pytest.raises(B.MpcmmdError, match="bad inner-CEM sizes"):
        _handle(mods, monkeypatch, "laplace", _args(5), 1, num_samples_cem=MAX_S + 1, maxiter_beta_cem=2)


@gpu
@pytest.mark.parametrize("ker,nr,S,mode", REF_CASES)
def test_generic_builds(mods, gk, monkeypatch, ker, nr, S, mode):
    """num_reduced 6..10: the generic kernel with the reference's sizes as template constants (S = 100) and with run-time sizes"""
    n = 3
    prob = _handle(mods, monkeypatch, ker, _args(nr), n, mode, num_samples_cem=S, maxiter_beta_cem=3)
    ora = _oracle(mods, gk, ker, _args(nr), num_samples_cem=S, maxiter_beta_cem=3)
    inp = _inputs(mods, ora, n, 10 * nr + S)
    got = _launch(f"ref/{ker}/{nr}/{S}/{mode}", lambda: _stage(prob, inp))
    _check(got, _refs(ora, inp, range(n)), f"nr={nr} S={S} {ker} {mode}")
    assert np.any(got["risk"] != f32(-1000.0))


# ---------------------------------------------------------------------------------------------------------------------------------
# automatic choice from the launch size

@gpu
@pytest.mark.parametrize("ker", ["laplace", "gaussian"])
def test_auto_dispatch_boundaries(mods, gk, monkeypatch, sms, ker):
    """nr 5, launches of SMs, SMs + 1, 3 SMs and 3 SMs + 1 chains: k_inner_cem_lat, the latency build twice, then the throughput build.
    Every chain of each launch equals the same chain from launches of at most SMs chains (k_inner_cem_lat), and a strided subset with the
    chains either side of each boundary equals the oracle"""
    S = AUTO_S[ker]
    n = 3 * sms + 1
    prob = _handle(mods, monkeypatch, ker, _args(5), n, num_samples_cem=S, maxiter_beta_cem=4)
    ora = _oracle(mods, gk, ker, _args(5), num_samples_cem=S, maxiter_beta_cem=4)
    inp = _inputs(mods, ora, n, 7)
    small = _launch(f"auto/{ker}/parts", lambda: _parts(prob, inp, n, sms))
    sizes = dict(zip(AUTO_POINTS, (sms, sms + 1, 3 * sms, 3 * sms + 1)))
    for p, m in sizes.items():
        got = _launch(f"auto/{ker}/{p}", lambda: _stage(prob, inp, 0, m))
        _same(got, {k: v[:m] for k, v in small.items()}, f"{ker} {m} chains in one launch vs launches of <= {sms}")
    _check(small, _refs(ora, inp, _strided(n, (sms - 1, sms, 3 * sms - 1, 3 * sms))), f"{ker} auto")
    assert len(np.unique(small["res_beta"][:, -1])) > n // 4


@gpu
@pytest.mark.parametrize("ker", ["laplace", "gaussian"])
def test_auto_dispatch_fast_math(mods, gk, monkeypatch, sms, ker):
    """MPCMMD_MATH=fast only changes the throughput build: 3 SMs chains still run the exact latency build, bit for bit, and 3 SMs + 1 run
    the fast-math build, within its tolerance"""
    S = AUTO_S[ker]
    n = 3 * sms + 1
    prob = _handle(mods, monkeypatch, ker, _args(5), n, fast_math=True, num_samples_cem=S, maxiter_beta_cem=4)
    ora = _oracle(mods, gk, ker, _args(5), num_samples_cem=S, maxiter_beta_cem=4)
    inp = _inputs(mods, ora, n, 8)
    exact = _launch(f"auto_fm/{ker}/3sm", lambda: _stage(prob, inp, 0, 3 * sms))
    fm = _launch(f"auto_fm/{ker}/3sm+1", lambda: _stage(prob, inp, 0, n))
    refs = _refs(ora, inp, _strided(n, (0, 3 * sms - 1, 3 * sms)))
    _check(exact, {i: r for i, r in refs.items() if i < 3 * sms}, f"{ker} fast math, 3 SMs chains")
    for i, ref in refs.items():
        _close({k: v[i] for k, v in fm.items()}, ref, f"{ker} fast math, {n} chains: chain {i}")


@gpu
@pytest.mark.parametrize("ker", ["laplace", "gaussian"])
def test_inner_cem_big_launch_shapes(mods, gk, monkeypatch, sms, ker):
    """nr 11: SMs chains run the 1024-thread build of k_inner_cem_big, SMs + 1 the 256-thread build; both equal each other chain for chain
    and a strided subset equals the oracle"""
    nr, n = 11, sms + 1
    kw = dict(num_samples_cem=40, maxiter_beta_cem=2)
    prob = _handle(mods, monkeypatch, ker, _args(nr), n, **kw)
    ora = _oracle(mods, gk, ker, _args(nr), **kw)
    inp = _inputs(mods, ora, n, 11)
    one = _launch(f"big/{ker}/sm", lambda: _stage(prob, inp, 0, sms))
    got = _launch(f"big/{ker}/sm+1", lambda: _stage(prob, inp, 0, n))
    _same({k: v[:sms] for k, v in got.items()}, one, f"{ker} nr=11: {n} chains (256 threads) vs {sms} (1024 threads)")
    _check(got, _refs(ora, inp, _strided(n, (sms - 1, sms), 6)), f"{ker} nr=11")


# ---------------------------------------------------------------------------------------------------------------------------------
# fast-math builds

@gpu
@pytest.mark.parametrize("ker,nr,S", FM_CASES)
def test_fast_math_build(mods, gk, monkeypatch, ker, nr, S):
    """MPCMMD_MATH=fast with the throughput build forced: the exponentials on MUFU.EX2, within the fast-math tolerance of the exact oracle"""
    n = 4
    kw = dict(num_samples_cem=S, maxiter_beta_cem=3)
    prob = _handle(mods, monkeypatch, ker, _args(nr), n, "cta", fast_math=True, **kw)
    ora = _oracle(mods, gk, ker, _args(nr), **kw)
    inp = _inputs(mods, ora, n, 20 + nr)
    got = _launch(f"fm/{ker}/{nr}/{S}", lambda: _stage(prob, inp))
    for i, ref in _refs(ora, inp, range(n)).items():
        _close({k: v[i] for k, v in got.items()}, ref, f"fast math {ker} nr={nr} S={S} chain {i}")


# ---------------------------------------------------------------------------------------------------------------------------------
# full solves

def _batch(O, ora, E):
    eps = [O.static_episode(2, k) for k in range(E)]
    tr = [ora.compute_obs_trajectories(*sc) for sc, _ in eps]
    init_state, mean, cov, v_des = O.driver_inputs("static")
    return dict(idx_mpc=[i for _, i in eps], init_state=np.stack([init_state] * E), mean_param=np.stack([mean] * E),
                cov_param=np.stack([cov] * E), x_obs_traj=np.stack([t[0] for t in tr]), y_obs_traj=np.stack([t[1] for t in tr]), v_des=[v_des] * E)


@gpu
@pytest.mark.parametrize("cell", list(SOLVE_CASES))
def test_solve(mods, gk, monkeypatch, sms, cell):
    """two episodes through the solve graph, which launches the same instantiation as a stage of that many chains, against the oracle's solve"""
    cem_impl, O = mods
    ker, nr, S, iters, B = SOLVE_CASES[cell]
    B = {"sm": sms, "2sm": 2 * sms}.get(B, B)
    E = 2
    kw = dict(num_batch=B, maxiter_cem=2, num_samples_cem=S, maxiter_beta_cem=iters)
    args = (nr, 2, 0.1, 30, "gaussian", 0.02, 0.01)
    monkeypatch.delenv("MPCMMD_INNER_CEM", raising=False)
    monkeypatch.delenv("MPCMMD_MATH", raising=False)
    prob = cem_impl.CEM(*args, max_episodes=E, kernel=ker, **kw)
    ora = _oracle(mods, gk, ker, args, **kw)
    b = _batch(O, ora, E)
    got = _launch(cell, lambda: prob.solve_batch("mmd_opt", **b))
    with ThreadPoolExecutor(max_workers=E) as ex:
        refs = list(ex.map(lambda e: ora.solve("mmd_opt", b["idx_mpc"][e], b["init_state"][e], b["mean_param"][e], b["cov_param"][e],
                                                b["x_obs_traj"][e], b["y_obs_traj"][e], b["v_des"][e]), range(E)))
    for e, ref in enumerate(refs):
        for k in SOLVE_KEYS:
            _eq(got[k][e], ref[k], f"{cell} episode {e} {k}")
    assert np.isfinite(got["res_beta"]).all() and got["res_beta"].shape == (E, iters)
