// k_validate_noise.cuh -- the noise half of `compute_stats` on the device: each trajectory's perturbed controls drawn from its own
// np.random.seed(key) stream (S/validation.py:40-90 = mpcmmd_b200.validation.perturbed_controls), for k_validate to roll out.
//
// A stream is sequential by definition (where each draw sits depends on every earlier rejection), so one thread consumes one stream.
// Each stream gets a 32-thread CTA of its own: the few hundred streams of a sweep point then spread over all SMs and their schedulers
// instead of sharing warps.  The 624-word MT19937 key lives in shared memory; lane 0 draws, twists and stores.
//
// Order and arithmetic (DESIGN.md section 3 item 6): beta noise draws beta(a|acc|, b|acc|, (n_roll, np)), beta(a|steer| + 1e-5,
// b|steer| + 1e-5, (n_roll, np)), multivariate_normal(0, I, (n_roll,)); Gaussian noise three multivariate_normal(0, I, (n_roll,)).
// multivariate_normal(0, I) is standard_normal in row-major order plus the mean 0.0.  The first two sections store plan +
// perturbation into acc / steer, the z section adds c * z to them: (plan + pert) + c * z, float64, no FMA.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "dnprng.cuh"

#define VALN_THREADS 32
#define VALN_STATE_WORDS (dnp::N + 4)        // key[624], pos, has_gauss, cached gauss (float64 bits, low word first)

struct ValNoiseCfg {
    int n_roll, np, noise_kind;               // noise_kind 0 gaussian, 1 beta
    double nl, k_steer, beta_a, beta_b, c_acc, c_steer;
};

// grid = trajectories.  seed (n,); acc_plan, steer_plan (n, np); acc, steer (n, n_roll, np) out; state_out (n, VALN_STATE_WORDS) or null
__global__ void __launch_bounds__(VALN_THREADS) k_validate_noise(ValNoiseCfg c, const uint32_t* __restrict__ seed,
                                                                 const double* __restrict__ acc_plan, const double* __restrict__ steer_plan,
                                                                 double* __restrict__ acc, double* __restrict__ steer,
                                                                 uint32_t* __restrict__ state_out) {
    __shared__ uint32_t key[dnp::N];
    if (threadIdx.x != 0) return;
    const int e = blockIdx.x, np = c.np;
    const double* ap = acc_plan + (size_t)e * np;
    const double* sp = steer_plan + (size_t)e * np;
    double* ao = acc + (size_t)e * c.n_roll * np;
    double* so = steer + (size_t)e * c.n_roll * np;
    dnp::State s; s.key = key;
    dnp::seed(s, seed[e]);
    if (c.noise_kind == 1) {
        for (int r = 0; r < c.n_roll; r++)
            for (int t = 0; t < np; t++)
                ao[(size_t)r * np + t] = ap[t] + c.nl * (2.0 * dnp::beta(s, c.beta_a * fabs(ap[t]), c.beta_b * fabs(ap[t])) - 1.0);
        const double ks = c.k_steer * c.nl;
        for (int r = 0; r < c.n_roll; r++)
            for (int t = 0; t < np; t++)
                so[(size_t)r * np + t] = sp[t] + ks * (2.0 * dnp::beta(s, c.beta_a * fabs(sp[t]) + 1e-5, c.beta_b * fabs(sp[t]) + 1e-5) - 1.0);
    } else {
        for (int r = 0; r < c.n_roll; r++)
            for (int t = 0; t < np; t++)
                ao[(size_t)r * np + t] = ap[t] + (c.nl * fabs(ap[t])) * (dnp::gauss(s) + 0.0);
        for (int r = 0; r < c.n_roll; r++)
            for (int t = 0; t < np; t++)
                so[(size_t)r * np + t] = sp[t] + (c.nl * fabs(sp[t])) * (dnp::gauss(s) + 0.0);
    }
    for (int r = 0; r < c.n_roll; r++)
        for (int t = 0; t < np; t++) {
            const double z = dnp::gauss(s) + 0.0;
            const size_t i = (size_t)r * np + t;
            ao[i] = ao[i] + c.c_acc * z;
            so[i] = so[i] + c.c_steer * z;
        }
    if (state_out) {
        uint32_t* w = state_out + (size_t)e * VALN_STATE_WORDS;
        for (int i = 0; i < dnp::N; i++) w[i] = key[i];
        const unsigned long long g = (unsigned long long)__double_as_longlong(s.gauss);
        w[dnp::N] = (uint32_t)s.pos; w[dnp::N + 1] = (uint32_t)s.has_gauss;
        w[dnp::N + 2] = (uint32_t)g; w[dnp::N + 3] = (uint32_t)(g >> 32);
    }
}
