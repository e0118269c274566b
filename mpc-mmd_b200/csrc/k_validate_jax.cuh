// k_validate_jax.cuh -- Monte-Carlo validation with counter-based noise (DESIGN.md section 3 item 7): the JAX-protocol draws
// (csrc/drng.cuh) are made by the thread that rolls the sample out, at the knot that consumes them, so no noise array exists and any
// number of rollouts per plan runs in one launch.
//
// Trajectory i with seed k: (k_acc, k_steer, k_z) = split(PRNGKey(k), 3).  Element e = r * np + t of n = n_roll * np:
//   beta noise      b_acc = beta(k_acc, f32(beta_a |acc_t|), f32(beta_b |acc_t|)), b_steer = beta(k_steer, f32(beta_a |steer_t| + 1e-5),
//                   f32(beta_b |steer_t| + 1e-5)); acc = (acc_t + nl (2 b_acc - 1)) + c_acc z, steer = (steer_t + K_steer nl (2 b_steer - 1)) + c_steer z
//   Gaussian noise  acc = (acc_t + (nl |acc_t|) z_acc) + c_acc z, steer likewise with z_steer; z_acc, z_steer = normal(k_acc), normal(k_steer)
//   z = normal(k_z).  Float32 draws widened exactly, float64 perturbation with validation.perturbed_controls' expressions (no FMA).
// A rollout's draws depend on n_roll (JAX lays the counters of the whole (n_roll, np) array out at once).
//
// grid = (rollout chunk, trajectory): thread tid of chunk b owns rollout b * VALJ_THREADS + tid, so one plan's 10^5 rollouts fill the GPU.
// Lanes of a warp are rollouts at the same knot: they share the Gamma shapes, only the rejection rounds diverge.  Each CTA counts into
// shared cnt[(O + 2)][np] (k_validate's layout and val_count) and adds them to the trajectory's global counters; k_validate_finish
// then reduces each trajectory as k_validate does.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "drng.cuh"
#include "k_validate.cuh"

#define VALJ_THREADS 256

struct ValJaxCfg {
    int noise_kind;                            // 0 gaussian, 1 beta
    double nl, ks, beta_a, beta_b, c_acc, c_steer;   // ks = K_steer * noise_level
};

// seed (n_ep,); acc_plan, steer_plan (n_ep, np); state0, x_obs, y_obs as k_validate; cnt_g (n_ep, O + 2, np) zeroed;
// acc_out, steer_out (n_ep, n_roll, np) the perturbed controls, or null.  Trajectory e = e0 + blockIdx.y.
// RISK: c_obs, c_lane (gridDim.y, n_roll) -- indexed by blockIdx.y, not e -- receive each rollout's obstacle and lane costs (as k_validate<true>).
template <bool RISK>
__global__ void __launch_bounds__(VALJ_THREADS) k_validate_jax(ValCfg c, ValJaxCfg j, int e0, const uint32_t* __restrict__ seed,
                                                               const double* __restrict__ acc_plan, const double* __restrict__ steer_plan,
                                                               const double* __restrict__ state0, const double* __restrict__ x_obs,
                                                               const double* __restrict__ y_obs, int32_t* __restrict__ cnt_g,
                                                               double* __restrict__ acc_out, double* __restrict__ steer_out,
                                                               double* __restrict__ c_obs, double* __restrict__ c_lane) {
    extern __shared__ int cnt[];
    const int e = e0 + blockIdx.y, tid = threadIdx.x, lane = tid & 31;
    const int np = c.np, O = c.O;
    for (int i = tid; i < (O + 2) * np; i += VALJ_THREADS) cnt[i] = 0;
    __syncthreads();
    const double* xo = x_obs + (size_t)e * O * np;
    const double* yo = y_obs + (size_t)e * O * np;
    const double* s0 = state0 + (size_t)e * 5;
    const double* ap = acc_plan + (size_t)e * np;
    const double* sp = steer_plan + (size_t)e * np;
    const int r = blockIdx.x * VALJ_THREADS + tid;
    const bool live = r < c.n_roll;
    const uint32_t n = (uint32_t)c.n_roll * (uint32_t)np;
    dr::Key k_acc, k_steer, k_z, ka_acc, kb_acc, ka_steer, kb_steer;
    dr::split3(dr::Key{0u, seed[e]}, k_acc, k_steer, k_z);
    if (j.noise_kind == 1) { dr::split2(k_acc, ka_acc, kb_acc); dr::split2(k_steer, ka_steer, kb_steer); }
    const size_t row = ((size_t)e * c.n_roll + (live ? r : 0)) * np;
    double x = s0[0], y = s0[1], vx = s0[2], vy = s0[3], psi = s0[4];
    ValRisk rk = {0.0, 0.0, 0.0};
    for (int t = 0; t < np; t++) {
        if constexpr (RISK) val_count<true>(c, xo, yo, t, x, y, live, lane, cnt, &rk);
        else val_count(c, xo, yo, t, x, y, live, lane, cnt);
        double a = 0.0, st = 0.0;
        if (live) {
            const uint32_t el = (uint32_t)r * (uint32_t)np + (uint32_t)t;
            const double pa = ap[t], ps = sp[t];
            if (j.noise_kind == 1) {
                const float ba = dr::beta_elem_split(ka_acc, kb_acc, n, el, (float)(j.beta_a * fabs(pa)), (float)(j.beta_b * fabs(pa)));
                const float bs = dr::beta_elem_split(ka_steer, kb_steer, n, el, (float)(j.beta_a * fabs(ps) + 1e-5), (float)(j.beta_b * fabs(ps) + 1e-5));
                a = pa + j.nl * (2.0 * (double)ba - 1.0);
                st = ps + j.ks * (2.0 * (double)bs - 1.0);
            } else {
                a = pa + (j.nl * fabs(pa)) * (double)dr::normal_elem(k_acc, n, el);
                st = ps + (j.nl * fabs(ps)) * (double)dr::normal_elem(k_steer, n, el);
            }
            const double z = (double)dr::normal_elem(k_z, n, el);
            a = a + j.c_acc * z;
            st = st + j.c_steer * z;
            if (acc_out) { acc_out[row + t] = a; steer_out[row + t] = st; }
        }
        val_step(c, a, st, x, y, vx, vy, psi);
    }
    if (RISK && live) {
        const size_t i = (size_t)blockIdx.y * c.n_roll + r;
        c_obs[i] = rk.obs; c_lane[i] = rk.lb + rk.ub;
    }
    __syncthreads();
    int32_t* g = cnt_g + (size_t)e * (O + 2) * np;
    for (int i = tid; i < (O + 2) * np; i += VALJ_THREADS)
        if (cnt[i]) atomicAdd(&g[i], cnt[i]);
}

// grid = trajectories, one warp each: the per-trajectory counters of k_validate_jax reduced as k_validate reduces its shared ones
__global__ void __launch_bounds__(32) k_validate_finish(int O, int np, const int32_t* __restrict__ cnt_g, int32_t* __restrict__ count,
                                                        int32_t* __restrict__ count_lane) {
    const int e = blockIdx.x;
    val_reduce(cnt_g + (size_t)e * (O + 2) * np, O, np, threadIdx.x, count + e, count_lane + e);
}
