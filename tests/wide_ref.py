"""CPU reference of cvar / saa / mmd_random at any num_reduced: tests/wide_oracle/oracle_wide.c (the frozen oracle plus heap-array
restatements of cvar_cost, the risk stage and the solve) behind OracleCEM's call surface.  Shared by tests/test_wide_oracle.py (CPU) and
tests/test_wide_rollout_sets.py (GPU)."""
import ctypes as C
import os
import subprocess

import numpy as np

f32 = np.float32
HERE = os.path.dirname(os.path.abspath(__file__))
KERNELS = {"laplace": 0, "gaussian": 1}


def build_lib(out_dir):
    """oracle_wide.c built with the oracle's flags into out_dir"""
    out = os.path.join(str(out_dir), "liboracle_wide.so")
    subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math", "-pthread",
                           "-Wall", "-Wno-unused-function", "-Wno-misleading-indentation", "-Wno-maybe-uninitialized",
                           os.path.join(HERE, "wide_oracle", "oracle_wide.c"), "-o", out, "-lm"])
    lib = C.CDLL(out)
    lib.oracle_set_threads(min(32, os.cpu_count() or 1))
    lib.wd_cvar.restype = C.c_float
    lib.wd_saa.restype = C.c_float
    return lib


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


class WRiskOut(C.Structure):
    _fields_ = [("risk", C.c_float), ("lane", C.c_float), ("sigma", C.c_float), ("beta", C.POINTER(C.c_float)), ("red_cost", C.POINTER(C.c_float))]


class WSolveOut(C.Structure):
    _fields_ = [("cx", C.c_float * 11), ("cy", C.c_float * 11), ("cost_lane", C.c_float), ("cost_obs", C.c_float), ("sigma", C.c_float),
                ("sel_last", C.c_int32)]


def cvar(lib, v, alpha=0.98):
    v = np.ascontiguousarray(v, f32)
    return f32(lib.wd_cvar(C.c_float(alpha), _fp(v), int(v.size)))


def saa(lib, v):
    v = np.ascontiguousarray(v, f32)
    return f32(lib.wd_saa(_fp(v), int(v.size)))


class WideOracle:
    """OracleCEM (constants, projection, noise tables, scene helpers) whose risk stage and solve, for cvar / saa / mmd_random, take any
    num_reduced.  The OracleCEM underneath is built at num_reduced 2 and then given num_reduced: only mmd_opt reads the tables that depend on
    it at construction (theta0, zb_iter, num_reduced^2 + 1 columns), and those are never used here."""

    def __init__(self, O, lib, num_reduced, *args, kernel="laplace", **kw):
        self._O, self._lib, self.kernel = O, lib, kernel
        ora = O.OracleCEM(2, *args, **kw)
        nr, nm = int(num_reduced), int(num_reduced) ** 2
        c = ora.cfg
        c.nr, c.nm = nr, nm
        c.inv_nm, c.m2_inv_nm = 1 / nm, -2 * (1 / nm)          # as OracleCEM.__init__ computes them
        c.beta_del = 1 / nr
        ora.num_reduced, ora.num_mother = nr, nm
        self._ora = ora

    def __getattr__(self, name):
        return getattr(self._ora, name)

    def risk(self, cost, acc, steer, st0, noise, x_obs_traj, y_obs_traj, beta_draws=None):
        O, ora, nr = self._O, self._ora, self._ora.num_reduced
        assert cost != "mmd_opt"
        z1, z2, z3, _, keys = noise
        b1 = b2 = None
        if beta_draws is not None:
            b1, b2 = (np.ascontiguousarray(b, f32).reshape(-1) for b in beta_draws)
        nz = O.ONoise(_fp(z1), _fp(z2), _fp(z3), (C.c_uint32 * 2)(keys[0], keys[1]), (C.c_uint32 * 2)(keys[2], keys[3]),
                      _fp(b1) if b1 is not None else None, _fp(b2) if b2 is not None else None)
        beta = np.zeros(nr, f32); red = np.zeros(nr, f32)
        o = WRiskOut(0.0, 0.0, 0.0, _fp(beta), _fp(red))
        acc = np.ascontiguousarray(acc, f32); steer = np.ascontiguousarray(steer, f32); st0 = np.ascontiguousarray(st0, f32)
        xo = np.ascontiguousarray(x_obs_traj, f32); yo = np.ascontiguousarray(y_obs_traj, f32)
        self._lib.wd_risk(ora._cfg_for(cost), KERNELS[self.kernel], O.COST_KINDS[cost], _fp(acc), _fp(steer), _fp(st0), C.byref(nz),
                          _fp(xo), _fp(yo), C.byref(o))
        return dict(risk=f32(o.risk), lane=f32(o.lane), beta=beta, sigma=f32(o.sigma), red_cost=red)

    def solve(self, cost, idx_mpc, init_state, mean, cov, x_obs_traj, y_obs_traj, v_des):
        O, ora, nr = self._O, self._ora, self._ora.num_reduced
        init_state = np.ascontiguousarray(init_state, f32); mean = np.ascontiguousarray(mean, f32)
        cov = np.ascontiguousarray(cov, f32); xo = np.ascontiguousarray(x_obs_traj, f32); yo = np.ascontiguousarray(y_obs_traj, f32)
        out = WSolveOut(); beta = np.zeros(nr, f32)
        self._lib.wd_solve(ora._cfg_for(cost), KERNELS[self.kernel], O.COST_KINDS[cost], C.c_int32(int(idx_mpc)), _fp(init_state), _fp(mean),
                           _fp(cov), _fp(xo), _fp(yo), C.c_float(v_des), C.byref(out), _fp(beta))
        return dict(cx=np.array(out.cx, f32), cy=np.array(out.cy, f32), cost_lane=f32(out.cost_lane), cost_obs=f32(out.cost_obs),
                    beta=beta, sigma=f32(out.sigma), sel=int(out.sel_last))
