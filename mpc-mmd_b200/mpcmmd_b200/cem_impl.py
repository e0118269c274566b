"""Drop-in `CEM` class: the reference's trajectory-optimizer call surface
(synthetic_static_obs/optimizer/cem.py:16-714) in front of libmpcmmd.so.

Same constructor, same four `compute_cem_*` methods (same argument meaning and return tuples), the
attributes `main_mpc.py` / `validation.py` read, plus a batched entry point (`solve_batch`) that
runs many independent episodes in one call -- the form the B200 kernels are built for.
PyTorch is used only to own device memory and the CUDA stream.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import binding as B
from .constants import NUM, NVAR, T_FIN, VARIANT_CONSTANTS, build_constants

F32 = np.float32


def _fp(a: np.ndarray):
    return a.ctypes.data_as(B.FP)


class _HelperShim:
    """The two members of `cem_helper.Helper` that callers touch (validation.py:151, main_mpc.py:109)."""

    def __init__(self, owner: "CEM"):
        self._o = owner
        self.K_steer = owner._K_steer                       # cem_helper.py:24

    def compute_obs_trajectories(self, x_obs, y_obs, vx_obs, vy_obs, psi_obs):
        """Constant-velocity obstacle tracks on tot_time (cem_helper.py:366-378); float32 like jnp."""
        tt = self._o.tot_time.astype(F32)[:, None]
        x = (np.asarray(x_obs, F32) + np.asarray(vx_obs, F32) * tt).T
        y = (np.asarray(y_obs, F32) + np.asarray(vy_obs, F32) * tt).T
        psi = np.tile(np.asarray(psi_obs, F32), (self._o.num, 1)).T
        return np.ascontiguousarray(x), np.ascontiguousarray(y), np.ascontiguousarray(psi)


class CEM:
    """`CEM(num_reduced, num_obs, noise_level, num_prime, noise, acc_const_noise, steer_const_noise)`
    (cem.py:17-18).  Keyword-only extras: `variant` ("static" | "dynamic": which of the reference's two
    optimizer/ copies to mirror), `max_episodes` (workspace capacity of `solve_batch`), `device`,
    `num_batch` / `maxiter_cem` overrides for scaled or reduced runs, `kernel` ("laplace" as the reference, or
    "gaussian"): the kernel of the MMD risk costs of mmd_opt and mmd_random, fixed for the object's lifetime
    (DESIGN.md section 3 items 4 and 8).
    `num_reduced` is 2..1024 for cvar, saa and mmd_random (above 64 one CTA per sample finishes the risk) and 2..40 for mmd_opt, whose
    solves and stages refuse larger sets; `tables()` (the mmd_opt inner-CEM tables) is refused above 64."""

    def __init__(self, num_reduced, num_obs, noise_level, num_prime, noise, acc_const_noise, steer_const_noise, *,
                 variant="static", max_episodes=1, device=0, num_batch=100, maxiter_cem=20,
                 num_samples_cem=100, maxiter_beta_cem=20, kernel="laplace"):
        if kernel not in B.MMD_KERNELS:
            raise ValueError(f"kernel must be one of {sorted(B.MMD_KERNELS)}, got {kernel!r}")
        self.kernel = kernel
        if noise not in B.NOISE_KINDS:
            noise_kind = B.NOISE_KINDS["beta"]               # reference: anything but "gaussian" takes the beta branch (cem_helper.py:405,416)
        else:
            noise_kind = B.NOISE_KINDS[noise]
        vc = VARIANT_CONSTANTS[variant]
        self.variant = variant
        # ---- attributes of the reference object (cem.py:20-171)
        self.acc_const_noise, self.steer_const_noise = acc_const_noise, steer_const_noise
        self.noise = noise
        self.beta_a, self.beta_b = 2, 5
        self.a_obs, self.b_obs = 4.25, 2.75
        self.wheel_base = 2.5
        self.v_max, self.v_min, self.a_max = 30.0, 0.1, 18.0
        self.num_obs = num_obs
        self.steer_max = 0.6
        self.t_fin, self.num = T_FIN, NUM
        self.t = self.t_fin / self.num
        self.num_prime = num_prime
        self.num_batch, self.maxiter_cem = num_batch, maxiter_cem
        self.ellite_num, self.ellite_num_cost = 5, min(20, num_batch)
        self.num_reduced, self.num_mother = num_reduced, num_reduced ** 2
        self.y_lb, self.y_ub = vc["y_lb"], vc["y_ub"]
        self._K_steer = vc["K_steer"]
        self.alpha_quant = 0.98
        self.ker_wt = 1000.0
        self.sigma_acc = self.sigma_steer = noise_level
        self.alpha_mean = self.alpha_cov = 0.6
        self.lamda = 0.9
        hc = build_constants(num_prime)
        self._hc = hc
        self.tot_time = hc.tot_time
        self.P, self.Pdot, self.Pddot = hc.P64, hc.Pdot64, hc.Pddot64           # NumPy float64, as in cem.py:46
        self.P_jax, self.Pdot_jax, self.Pddot_jax = hc.P, hc.Pdot, hc.Pddot     # float32 (jnp.asarray), cem.py:48
        self.nvar = NVAR
        self.cem_helper = _HelperShim(self)
        self.num_samples_cem, self.maxiter_beta_cem = num_samples_cem, maxiter_beta_cem
        self.num_ellite_beta = max(int(0.1 * num_samples_cem) + 1, 3)            # compute_beta.py:26

        # ---- device handle
        import torch
        if not torch.cuda.is_available():
            raise B.MpcmmdError("CEM needs a CUDA device: the B200 kernels have no CPU fallback")
        self._torch = torch
        self.device = torch.device("cuda", device)
        self.max_episodes = int(max_episodes)
        cfg = B.MpcmmdConfig()
        cfg.num_batch, cfg.num_prime, cfg.num_reduced, cfg.num_obs = num_batch, num_prime, num_reduced, num_obs
        cfg.maxiter_cem, cfg.ellite_num, cfg.ellite_num_cost = maxiter_cem, self.ellite_num, self.ellite_num_cost
        cfg.noise_kind = noise_kind
        cfg.num_samples_cem, cfg.maxiter_beta_cem, cfg.num_ellite_beta = num_samples_cem, maxiter_beta_cem, self.num_ellite_beta
        cfg.max_episodes = self.max_episodes
        cfg.sigma_acc = cfg.sigma_steer = noise_level
        cfg.ksig_steer = self._K_steer * noise_level            # double product, then float32 (cem_helper.py:436)
        cfg.acc_const_noise, cfg.steer_const_noise = acc_const_noise, steer_const_noise
        cfg.beta_a, cfg.beta_b = self.beta_a, self.beta_b
        cfg.v_min, cfg.v_max, cfg.a_max = self.v_min, self.v_max, self.a_max
        cfg.y_lb, cfg.y_ub = self.y_lb, self.y_ub
        cfg.a_obs_sq, cfg.b_obs_sq = self.a_obs ** 2, self.b_obs ** 2
        cfg.wheel_base, cfg.dt, cfg.steer_max, cfg.steer_rate_pen = self.wheel_base, self.t, self.steer_max, 0.05
        cfg.alpha_quant, cfg.ker_wt = self.alpha_quant, self.ker_wt
        cfg.lamda_inv = 1 / self.lamda
        cfg.alpha_mean, cfg.alpha_cov = self.alpha_mean, self.alpha_cov
        cfg.one_minus_alpha_mean, cfg.one_minus_alpha_cov = 1 - self.alpha_mean, 1 - self.alpha_cov
        cfg.sigma_clip, cfg.sigma_random = 0.01, 0.01
        cfg.P, cfg.Pdot, cfg.Pddot = _fp(hc.P), _fp(hc.Pdot), _fp(hc.Pddot)
        cfg.Gx, cfg.Gy, cfg.Kx, cfg.Ky, cfg.Wfit = _fp(hc.Gx), _fp(hc.Gy), _fp(hc.Kx), _fp(hc.Ky), _fp(hc.Wfit)
        self._cfg = cfg
        self._lib = B.load()
        self._h = C.c_void_p()
        B.check(self._lib.mpcmmd_create_with_kernel(C.byref(cfg), B.MMD_KERNELS[kernel], int(device), C.byref(self._h)))

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            self._lib.mpcmmd_destroy(h)
            self._h = C.c_void_p()

    # ------------------------------------------------------------------------------------------
    def _dev(self, a, dtype):
        torch = self._torch
        if isinstance(a, torch.Tensor):
            return a.to(device=self.device, dtype=dtype).contiguous()
        return torch.as_tensor(np.ascontiguousarray(np.asarray(a), dtype=np.int32 if dtype == torch.int32 else F32),
                               device=self.device)

    def solve_batch_device(self, cost, idx_mpc, init_state, mean_param, cov_param, x_obs_traj, y_obs_traj, v_des):
        """n_ep independent solves with inputs/outputs as CUDA tensors (no host copies).  Shapes:
        idx_mpc (E,), init_state (E,6), mean_param (E,8), cov_param (E,8,8), x/y_obs_traj (E,num_obs,100), v_des (E,).
        Returns a dict of CUDA tensors: cx, cy (E,11), cost_lane, cost_obs (E,), beta (E,nr), sigma (E,), res_beta (E,20)."""
        torch = self._torch
        kind = B.COST_KINDS[cost]
        idx = self._dev(idx_mpc, torch.int32)
        E = int(idx.shape[0])
        st = self._dev(init_state, torch.float32).reshape(E, 6)
        mean = self._dev(mean_param, torch.float32).reshape(E, 8)
        cov = self._dev(cov_param, torch.float32).reshape(E, 64)
        xo = self._dev(x_obs_traj, torch.float32).reshape(E, self.num_obs, NUM)
        yo = self._dev(y_obs_traj, torch.float32).reshape(E, self.num_obs, NUM)
        vd = self._dev(v_des, torch.float32).reshape(E)
        f = dict(device=self.device, dtype=torch.float32)
        out = dict(cx=torch.empty(E, NVAR, **f), cy=torch.empty(E, NVAR, **f), cost_lane=torch.empty(E, **f), cost_obs=torch.empty(E, **f),
                   beta=torch.empty(E, self.num_reduced, **f), sigma=torch.empty(E, **f), res_beta=torch.empty(E, self.maxiter_beta_cem, **f))
        o = B.MpcmmdOut(*[out[k].data_ptr() for k in ("cx", "cy", "cost_lane", "cost_obs", "beta", "sigma", "res_beta")])
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            B.check(self._lib.mpcmmd_solve(self._h, kind, E, idx.data_ptr(), st.data_ptr(), mean.data_ptr(), cov.data_ptr(), xo.data_ptr(),
                                           yo.data_ptr(), vd.data_ptr(), C.byref(o), C.c_void_p(stream)))
        out["_keepalive"] = (idx, st, mean, cov, xo, yo, vd)
        return out

    def solve_batch(self, cost, idx_mpc, init_state, mean_param, cov_param, x_obs_traj, y_obs_traj, v_des):
        """Host-array version of `solve_batch_device`: NumPy in, NumPy out (copies inside the library)."""
        kind = B.COST_KINDS[cost]
        idx = np.ascontiguousarray(np.asarray(idx_mpc), np.int32).reshape(-1)
        E = idx.shape[0]
        st = np.ascontiguousarray(np.asarray(init_state), F32).reshape(E, 6)
        mean = np.ascontiguousarray(np.asarray(mean_param), F32).reshape(E, 8)
        cov = np.ascontiguousarray(np.asarray(cov_param), F32).reshape(E, 64)
        xo = np.ascontiguousarray(np.asarray(x_obs_traj), F32).reshape(E, self.num_obs, NUM)
        yo = np.ascontiguousarray(np.asarray(y_obs_traj), F32).reshape(E, self.num_obs, NUM)
        vd = np.ascontiguousarray(np.asarray(v_des), F32).reshape(E)
        out = dict(cx=np.empty((E, NVAR), F32), cy=np.empty((E, NVAR), F32), cost_lane=np.empty(E, F32), cost_obs=np.empty(E, F32),
                   beta=np.empty((E, self.num_reduced), F32), sigma=np.empty(E, F32), res_beta=np.empty((E, self.maxiter_beta_cem), F32))
        o = B.MpcmmdOut(*[out[k].ctypes.data for k in ("cx", "cy", "cost_lane", "cost_obs", "beta", "sigma", "res_beta")])
        B.check(self._lib.mpcmmd_solve_host(self._h, kind, E, idx.ctypes.data, st.ctypes.data, mean.ctypes.data, cov.ctypes.data,
                                            xo.ctypes.data, yo.ctypes.data, vd.ctypes.data, C.byref(o)))
        return out

    def inner_cem_path(self) -> str:
        """name of the reduced-set inner-CEM kernel path a throughput-sized mmd_opt launch of this handle takes (reporting only)"""
        return self._lib.mpcmmd_inner_cem_path(self._h).decode()

    def last_launch_count(self) -> int:
        return int(self._lib.mpcmmd_last_launch_count(self._h))

    def profile_solve(self, cost, n_ep):
        """Device time per kernel class of the solve staged by the previous solve call (launch-by-launch CUDA events)."""
        ms = (C.c_float * 5)(); nl = (C.c_int * 4)()
        B.check(self._lib.mpcmmd_profile_solve(self._h, B.COST_KINDS[cost], int(n_ep), ms, nl))
        names = ("setup", "project", "risk", "select")
        return {"ms": dict(zip(names + ("total",), [float(v) for v in ms])), "launches": dict(zip(names, [int(v) for v in nl]))}

    def _single(self, cost, idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des):
        r = self.solve_batch(cost, [int(idx_mpc)], np.asarray(init_state, F32)[None], np.asarray(mean_param_init, F32)[None],
                             np.asarray(cov_param_init, F32)[None], np.asarray(x_obs_traj, F32)[None], np.asarray(y_obs_traj, F32)[None],
                             [float(v_des)])
        return {k: v[0] for k, v in r.items()}

    # ---- the reference's four entry points (cem.py:201-333, 335-462, 464-588, 590-714) ---------
    def compute_cem_mmd_opt(self, idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des):
        r = self._single("mmd_opt", idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des)
        return r["cx"], r["cy"], r["cost_lane"], r["cost_obs"], r["beta"], r["sigma"], r["res_beta"]

    def compute_cem_mmd_random(self, idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des):
        r = self._single("mmd_random", idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des)
        return r["cx"], r["cy"], r["cost_lane"], r["cost_obs"]

    def compute_cem_cvar(self, idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des):
        r = self._single("cvar", idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des)
        return r["cx"], r["cy"], r["cost_lane"], r["cost_obs"]

    def compute_cem_saa(self, idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des):
        r = self._single("saa", idx_mpc, init_state, mean_param_init, cov_param_init, x_obs_traj, y_obs_traj, v_des)
        return r["cx"], r["cy"], r["cost_lane"], r["cost_obs"]

    # ---- stage entry points (teacher-forced parity tests) -------------------------------------
    def _t(self, a, dtype=None):
        torch = self._torch
        dtype = dtype or torch.float32
        if dtype == torch.float32:
            return torch.as_tensor(np.ascontiguousarray(np.asarray(a), F32), device=self.device)
        return torch.as_tensor(np.ascontiguousarray(np.asarray(a)), device=self.device).to(dtype)

    def stage_project(self, params, beq_x, beq_y, v_des, lam_x, lam_y, s_lane):
        torch = self._torch
        p = self._t(params); n = p.shape[0]
        bx, by = self._t(beq_x), self._t(beq_y)
        lx, ly, sl = self._t(lam_x).clone(), self._t(lam_y).clone(), self._t(s_lane).clone()
        f = dict(device=self.device, dtype=torch.float32)
        o = dict(cx=torch.empty(n, NVAR, **f), cy=torch.empty(n, NVAR, **f), res_norm=torch.empty(n, **f), acc=torch.empty(n, NUM, **f),
                 steer=torch.empty(n, NUM, **f), cost_base=torch.empty(n, **f))
        B.check(self._lib.mpcmmd_stage_project(self._h, n, p.data_ptr(), bx.data_ptr(), by.data_ptr(), float(v_des), lx.data_ptr(), ly.data_ptr(),
                                               sl.data_ptr(), o["cx"].data_ptr(), o["cy"].data_ptr(), o["res_norm"].data_ptr(), o["acc"].data_ptr(),
                                               o["steer"].data_ptr(), o["cost_base"].data_ptr()))
        o.update(lam_x=lx, lam_y=ly, s_lane=sl)
        return {k: v.cpu().numpy() for k, v in o.items()}

    def stage_noise(self, idx_mpc, it):
        torch = self._torch
        n = self.num_reduced * self.num_prime
        f = dict(device=self.device, dtype=torch.float32)
        z1, z2, z3 = (torch.empty(n, **f) for _ in range(3))
        zc = torch.empty((self.num_batch - self.ellite_num) * 8, **f)
        keys = torch.empty(4, device=self.device, dtype=torch.int32)
        B.check(self._lib.mpcmmd_stage_noise(self._h, int(idx_mpc), int(it), z1.data_ptr(), z2.data_ptr(), z3.data_ptr(), zc.data_ptr(), keys.data_ptr()))
        return z1.cpu().numpy(), z2.cpu().numpy(), z3.cpu().numpy(), zc.cpu().numpy().reshape(-1, 8), [int(k) & 0xFFFFFFFF for k in keys.cpu().tolist()]

    def stage_risk(self, cost, acc, steer, state0, noise, x_obs_traj, y_obs_traj):
        torch = self._torch
        a, s = self._t(acc), self._t(steer); n = a.shape[0]
        z1, z2, z3, _, keys = noise
        st0 = self._t(state0)
        kz = torch.as_tensor(np.asarray(keys, dtype=np.uint32).view(np.int32), device=self.device)
        xo, yo = self._t(x_obs_traj), self._t(y_obs_traj)
        f = dict(device=self.device, dtype=torch.float32)
        o = dict(risk=torch.empty(n, **f), lane=torch.empty(n, **f), beta=torch.zeros(n, self.num_reduced, **f), sigma=torch.zeros(n, **f),
                 res_beta=torch.zeros(n, self.maxiter_beta_cem, **f))
        tz1, tz2, tz3 = self._t(z1), self._t(z2), self._t(z3)          # keep the tensors alive across the call
        B.check(self._lib.mpcmmd_stage_risk(self._h, B.COST_KINDS[cost], n, a.data_ptr(), s.data_ptr(), st0.data_ptr(), tz1.data_ptr(),
                                            tz2.data_ptr(), tz3.data_ptr(), kz.data_ptr(), xo.data_ptr(), yo.data_ptr(),
                                            o["risk"].data_ptr(), o["lane"].data_ptr(), o["beta"].data_ptr(), o["sigma"].data_ptr(), o["res_beta"].data_ptr()))
        return {k: v.cpu().numpy() for k, v in o.items()}

    def stage_risk_injected(self, cost, acc, steer, state0, z3, beta_acc, beta_steer, x_obs_traj, y_obs_traj):
        """risk stage with the beta-noise draws injected: beta_acc, beta_steer (n, nr*np) = the reference's jax.random.beta samples"""
        torch = self._torch
        a, s = self._t(acc), self._t(steer); n = a.shape[0]
        st0, tz3 = self._t(state0), self._t(z3)
        b1, b2 = self._t(np.asarray(beta_acc, F32).reshape(n, -1)), self._t(np.asarray(beta_steer, F32).reshape(n, -1))
        xo, yo = self._t(x_obs_traj), self._t(y_obs_traj)
        f = dict(device=self.device, dtype=torch.float32)
        o = dict(risk=torch.empty(n, **f), lane=torch.empty(n, **f), beta=torch.zeros(n, self.num_reduced, **f), sigma=torch.zeros(n, **f),
                 res_beta=torch.zeros(n, self.maxiter_beta_cem, **f))
        B.check(self._lib.mpcmmd_stage_risk_injected(self._h, B.COST_KINDS[cost], n, a.data_ptr(), s.data_ptr(), st0.data_ptr(), tz3.data_ptr(),
                                                     b1.data_ptr(), b2.data_ptr(), xo.data_ptr(), yo.data_ptr(), o["risk"].data_ptr(),
                                                     o["lane"].data_ptr(), o["beta"].data_ptr(), o["sigma"].data_ptr(), o["res_beta"].data_ptr()))
        return {k: v.cpu().numpy() for k, v in o.items()}

    def stage_init(self, mean, cov):
        """initial CEM batch (B,8) of `Helper.sampling_param` for (mean, cov)"""
        torch = self._torch
        m, cv = self._t(mean), self._t(np.asarray(cov, F32).reshape(-1))
        out = torch.empty(self.num_batch, 8, device=self.device, dtype=torch.float32)
        B.check(self._lib.mpcmmd_stage_init(self._h, m.data_ptr(), cv.data_ptr(), out.data_ptr()))
        return out.cpu().numpy()

    def stage_select(self, cost, res_norm, risk, cost_base, params, mean, cov, z_cem):
        torch = self._torch
        p = self._t(params).clone(); m = self._t(mean).clone(); cv = self._t(np.asarray(cov, F32).reshape(-1)).clone()
        sel = torch.zeros(1, device=self.device, dtype=torch.int32)
        tres, trisk, tbase, tz = self._t(res_norm), self._t(risk), self._t(cost_base), self._t(z_cem)
        B.check(self._lib.mpcmmd_stage_select(self._h, B.COST_KINDS[cost], tres.data_ptr(), trisk.data_ptr(), tbase.data_ptr(), p.data_ptr(),
                                              m.data_ptr(), cv.data_ptr(), tz.data_ptr(), sel.data_ptr()))
        return p.cpu().numpy(), m.cpu().numpy(), cv.cpu().numpy().reshape(8, 8), int(sel.item())

    def tables(self):
        torch = self._torch
        d = self.num_mother + 1
        f = dict(device=self.device, dtype=torch.float32)
        zi = torch.empty(self.num_batch, 8, **f); th = torch.empty(self.num_samples_cem, d, **f)
        zb = torch.empty(self.maxiter_beta_cem, self.num_samples_cem - self.num_ellite_beta, d, **f)
        B.check(self._lib.mpcmmd_get_tables(self._h, zi.data_ptr(), th.data_ptr(), zb.data_ptr()))
        return zi.cpu().numpy(), th.cpu().numpy(), zb.cpu().numpy()


# device-level primitives for the math / RNG parity tests
def math_vec(fn: int, x, y=None, device=0):
    import torch
    lib = B.load()
    xt = torch.as_tensor(np.ascontiguousarray(x, F32), device=f"cuda:{device}")
    yt = xt if y is None else torch.as_tensor(np.ascontiguousarray(y, F32), device=f"cuda:{device}")
    out = torch.empty_like(xt)
    B.check(lib.mpcmmd_math_vec(fn, xt.data_ptr(), yt.data_ptr(), out.data_ptr(), xt.numel(), device))
    return out.cpu().numpy()


def rng_normal(key, n, device=0):
    import torch
    lib = B.load()
    out = torch.empty(n, device=f"cuda:{device}", dtype=torch.float32)
    B.check(lib.mpcmmd_rng_normal(key[0], key[1], n, out.data_ptr(), device))
    return out.cpu().numpy()


def rng_beta(key, a, b, device=0):
    import torch
    lib = B.load()
    at = torch.as_tensor(np.ascontiguousarray(a, F32), device=f"cuda:{device}")
    bt = torch.as_tensor(np.ascontiguousarray(b, F32), device=f"cuda:{device}")
    out = torch.empty_like(at)
    B.check(lib.mpcmmd_rng_beta(key[0], key[1], at.data_ptr(), bt.data_ptr(), at.numel(), out.data_ptr(), device))
    return out.cpu().numpy()


def fp32_peak(device=0):
    """(TFLOP/s, SM count): FP32 FMA throughput measured by a register-resident fma micro-kernel."""
    lib = B.load()
    tf = C.c_float(); sm = C.c_int()
    B.check(lib.mpcmmd_fp32_peak(int(device), C.byref(tf), C.byref(sm)))
    return float(tf.value), int(sm.value)


def selfcheck_ieee(device=0):
    """(sqrt, reciprocal-of-sqrt, divide-by-10) mismatch counts of the device's IEEE shortcuts against sqrtf / division over all 2^32 float bit patterns."""
    lib = B.load()
    m = (C.c_ulonglong * 3)()
    B.check(lib.mpcmmd_selfcheck_ieee(int(device), m))
    return int(m[0]), int(m[1]), int(m[2])


def xu_peaks(device=0):
    """dict(ex2_gops, div_gops, sqrt_gops): measured MUFU.EX2 / IEEE division / IEEE square-root throughput (thread-level Gop/s)."""
    lib = B.load()
    g = (C.c_float * 3)()
    B.check(lib.mpcmmd_xu_peaks(int(device), g))
    return dict(ex2_gops=float(g[0]), div_gops=float(g[1]), sqrt_gops=float(g[2]))
