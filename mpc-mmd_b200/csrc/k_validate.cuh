// k_validate.cuh -- Monte-Carlo validation of a planned trajectory: the rollout + collision / lane counting part of
// `compute_stats` (reference S/validation.py:134-171 = compute_rollout_complete :40-105, compute_rollout_one_step :21-38,
// compute_f_bar_temp :107-114, compute_lane_bar :116-124; D/validation.py:129-165 likewise).  The reference draws its noise from
// NumPy's legacy MT19937 stream (np.random.seed(key); multivariate_normal / beta, S/validation.py:43-84): those draws stay on the
// host (bit-identical streams), the perturbed controls come in as float64 arrays and everything after them runs here.
//
// Arithmetic follows the reference's NumPy expression order in float64 (compiled with --fmad=false).  The obstacle cost is
// evaluated in float32 for the static variant -- there `x_obs_traj` is a float32 jax array (cem_helper.compute_obs_trajectories), so
// `x - x_obs` and everything downstream of it is float32 -- and in float64 for the dynamic variant (the trajectories are read back
// from the .npz as NumPy float64; D/validation.py:131-133).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define VAL_THREADS 256

struct ValCfg {
    int n_roll, np, O, obs_f32;
    double dt, wheel_base, a2, b2, y_lb, y_ub;
};

// Shared counters cnt[(O + 2)][np]: rows 0..O-1 obstacle intersections per (obstacle, timestep), row O lower-lane, row O+1 upper-lane
// violations per timestep.  val_count adds one rollout state per lane at timestep t; every lane of the warp must call it (ballots).
// xo, yo: the trajectory's obstacle trajectories (O, np).
// Risk statistics (DESIGN.md section 3 item 9): a rollout's running maxima of max(0, obstacle cost) over (obstacle, t) and of the two lane
// violations over t, NaN propagating as np.max(np.maximum(0, .)) does.  Only the RISK instantiations keep them.
struct ValRisk { double obs, lb, ub; };
__device__ __forceinline__ double val_nanmax(double m, double v) { return (v > m || v != v) ? v : m; }

template <bool RISK = false>
__device__ __forceinline__ void val_count(const ValCfg& c, const double* __restrict__ xo, const double* __restrict__ yo, int t, double x,
                                          double y, bool live, int lane, int* cnt, ValRisk* rk = nullptr) {
    const int np = c.np, O = c.O;
    const float a2f = (float)c.a2, b2f = (float)c.b2;
    for (int o = 0; o < O; o++) {
        bool nz;
        if (c.obs_f32) {
            const float wc = (float)x - (float)xo[o * np + t], ws = (float)y - (float)yo[o * np + t];
            const float cost = ((-(wc * wc)) / a2f - (ws * ws) / b2f) + 1.0f;          // S/validation.py:112
            nz = (cost > 0.0f) || (cost != cost);                                       // np.maximum(0, cost) != 0 (NaN counts)
            if (RISK) rk->obs = val_nanmax(rk->obs, (double)cost);                      // the float32 maximum, widened exactly
        } else {
            const double wc = x - xo[o * np + t], ws = y - yo[o * np + t];
            const double cost = ((-(wc * wc)) / c.a2 - (ws * ws) / c.b2) + 1.0;
            nz = (cost > 0.0) || (cost != cost);
            if (RISK) rk->obs = val_nanmax(rk->obs, cost);
        }
        const unsigned m = __ballot_sync(0xffffffffu, live && nz);
        if (lane == 0 && m) atomicAdd(&cnt[o * np + t], __popc(m));
    }
    const double lb = -y + c.y_lb, ub = y - c.y_ub;                                     // S/validation.py:118-119
    if (RISK) { rk->lb = val_nanmax(rk->lb, lb); rk->ub = val_nanmax(rk->ub, ub); }
    const unsigned ml = __ballot_sync(0xffffffffu, live && ((lb > 0.0) || (lb != lb)));
    const unsigned mu = __ballot_sync(0xffffffffu, live && ((ub > 0.0) || (ub != ub)));
    if (lane == 0 && ml) atomicAdd(&cnt[O * np + t], __popc(ml));
    if (lane == 0 && mu) atomicAdd(&cnt[(O + 1) * np + t], __popc(mu));
}

// one bicycle-model step with controls (a, st) (S/validation.py:21-38)
__device__ __forceinline__ void val_step(const ValCfg& c, double a, double st, double& x, double& y, double& vx, double& vy, double& psi) {
    double v = sqrt(vx * vx + vy * vy);
    v = v + a * c.dt;
    const double psidot = v * tan(st) / c.wheel_base;
    const double psi_next = psi + psidot * c.dt;
    const double vx_next = v * cos(psi_next), vy_next = v * sin(psi_next);
    x = x + vx_next * c.dt; y = y + vy_next * c.dt;
    vx = vx_next; vy = vy_next; psi = psi_next;
}

// one warp: count = max over (obstacle, timestep) of the intersection counts; count_lane = max_t lb + max_t ub (S/validation.py:156-169)
__device__ __forceinline__ void val_reduce(const int* cnt, int O, int np, int lane, int32_t* count, int32_t* count_lane) {
    int m = 0, l = 0, u = 0;
    for (int i = lane; i < O * np; i += 32) m = max(m, cnt[i]);
    for (int t = lane; t < np; t += 32) { l = max(l, cnt[O * np + t]); u = max(u, cnt[(O + 1) * np + t]); }
    for (int off = 16; off >= 1; off >>= 1) {
        m = max(m, __shfl_xor_sync(0xffffffffu, m, off)); l = max(l, __shfl_xor_sync(0xffffffffu, l, off)); u = max(u, __shfl_xor_sync(0xffffffffu, u, off));
    }
    if (lane == 0) { *count = m; *count_lane = l + u; }
}

// grid = episodes; thread r handles rollouts r, r + VAL_THREADS, ...  RISK: c_obs, c_lane (n_ep, n_roll) receive each rollout's obstacle and lane
// costs (DESIGN.md section 3 item 9); the counting is the same.  The two pointers come last, so RISK = false compiles to the counting-only
// kernel's instructions with the same parameter offsets.
template <bool RISK>
__global__ void __launch_bounds__(VAL_THREADS) k_validate(ValCfg c, const double* __restrict__ acc, const double* __restrict__ steer,
                                                          const double* __restrict__ state0, const double* __restrict__ x_obs,
                                                          const double* __restrict__ y_obs, int32_t* __restrict__ count,
                                                          int32_t* __restrict__ count_lane, double* __restrict__ x_roll, double* __restrict__ y_roll,
                                                          double* __restrict__ c_obs, double* __restrict__ c_lane) {
    extern __shared__ int cnt[];
    const int e = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
    const int np = c.np, O = c.O;
    for (int i = tid; i < (O + 2) * np; i += VAL_THREADS) cnt[i] = 0;
    __syncthreads();
    const double* xo = x_obs + (size_t)e * O * np;
    const double* yo = y_obs + (size_t)e * O * np;
    const double* s0 = state0 + (size_t)e * 5;
    for (int base = 0; base < c.n_roll; base += VAL_THREADS) {
        const int r = base + tid;
        const bool live = r < c.n_roll;
        const size_t row = ((size_t)e * c.n_roll + (live ? r : 0)) * np;
        double x = s0[0], y = s0[1], vx = s0[2], vy = s0[3], psi = s0[4];
        // the maxima live in shared memory: in registers they would be saved around the double trig slow-path call (local-memory spills)
        __shared__ ValRisk rks[VAL_THREADS];
        ValRisk& rk = rks[tid];
        if constexpr (RISK) rk = ValRisk{0.0, 0.0, 0.0};
        for (int t = 0; t < np; t++) {
            // ---- record the state before the step (S/validation.py:98-100) and count on it
            if (live && x_roll) { x_roll[row + t] = x; y_roll[row + t] = y; }
            if constexpr (RISK) val_count<true>(c, xo, yo, t, x, y, live, lane, cnt, &rk);
            else val_count(c, xo, yo, t, x, y, live, lane, cnt);
            val_step(c, live ? acc[row + t] : 0.0, live ? steer[row + t] : 0.0, x, y, vx, vy, psi);
        }
        if (RISK && live) { c_obs[row / np] = rk.obs; c_lane[row / np] = rk.lb + rk.ub; }
    }
    __syncthreads();
    if (tid < 32) val_reduce(cnt, O, np, lane, count + e, count_lane + e);
}
