// k_risk.cuh -- noisy control rollouts, reduced-set selection and the risk functionals.
//
// Replaces, per CEM sample:
//   Helper.compute_rollout_complete_baseline / _opt + compute_rollout_one_step   S/optimizer/cem_helper.py:402-538, 380-400
//   Helper.compute_coeff                                                         S/optimizer/cem_helper.py:553-564
//   beta_cem.compute_cem (+ compute_mean_cov_beta, compute_beta_reduced)          S/compute_beta.py:93-157, 51-91
//   kernel_matrix.compute_kernel / compute_mmd (Laplace kernel)                   S/kernel_computation.py:19-87
//   Costs.compute_f_bar / compute_lane_bar / compute_{mmd,cvar,saa}_{obs,lane}     S/optimizer/costs.py:50-71, 121-234
// k_rollouts<MODE>: noisy controls + rollouts; ROLL_OPT writes the mother samples' ridge-fit features and controls for the inner CEM,
//              ROLL_FLY / ROLL_STAGED finish cvar / saa / mmd_random (risk folded into the rollout / reduced by a warp per sample).
// k_inner_cem<NR>: generic reduced-set inner CEM, one CTA per sample with all state in shared memory (num_reduced 6..10, and the
//              reference for the kernel-variant tests); the production kernel for num_reduced <= 5 is k_inner_cem_fast (k_inner_cem.cuh).
#pragma once
#include "common.cuh"

struct RiskArgs {
    int n_samples, B, cost_kind;
    const float *acc, *steer;        // [n][100]
    const float* state0;             // [E][5]
    const float *z1, *z2, *z3;       // episode e at z + e*z_stride, (nr,np)
    size_t z_stride;
    const uint32_t* keys;            // episode e at keys + e*key_stride, 4 words
    size_t key_stride;
    const float* btab;               // episode e at btab + e*btab_stride: [4][GT_FIELDS][nr*np] (beta noise; null -> direct sampler)
    size_t btab_stride;
    const float *binj1, *binj2;      // [n][nr*np] injected Beta draws (acceleration, steering) instead of the device sampler; null in solves (mpcmmd_stage_risk_injected)
    const float *x_obs, *y_obs;      // [E][O][100]
    const float *sx_obs, *sy_obs;    // [E][100][O] sorted by x per knot, or null (plain obstacle loop)
    const int* obs_nan;              // [E][100]
    float *risk, *lane;              // [n]
    float *beta, *sigma, *res_beta;  // [n][nr], [n], [n][iters_in]
};

// obstacle indicator at one (rollout point, obstacle point)  [costs.py:50-60]
__device__ __forceinline__ float fbar(const DCfg& c, float x, float y, float xo, float yo) {
    float wc = x - xo, ws = y - yo;
    const float A = wc * wc, B = ws * ws;
    // exact screen: outside the obstacle's ellipse box the indicator is 0 without the two IEEE divisions.  A >= a^2 makes the rounded quotient
    // -A/a^2 <= -1 (rounding is monotone and -1 is representable), B/b^2 >= 0, so the rounded sum is <= -1 and cost <= 0 -> max0 = 0; the same with
    // the roles swapped.  NaN operands fail the screen and take the full path, so NaN propagation is unchanged.
    if (((A >= c.a2_obs) || (B >= c.b2_obs)) && A == A && B == B) return 0.0f;
    float cost = (-A / c.a2_obs - B / c.b2_obs) + 1.0f;
    return dm::max0_(cost);
}
// one step of the Euler bicycle model  [cem_helper.py:380-400]; `ts` = tan(steer).  The tangent does not depend on the state, so wherever the
// controls are staged it is taken there, in parallel and once per control element (a mother rollout shares its steering row with
// num_reduced - 1 others), instead of inside the serial per-step chain.
__device__ __forceinline__ void bicycle_step(const DCfg& c, float a, float ts, float& x, float& y, float& vx, float& vy, float& psi) {
    float v = sqrtf(vx * vx + vy * vy);
    v = v + a * c.dt;
    float psidot = (v * ts) / c.wheel_base;
    psi = psi + psidot * c.dt;
    float sp, cp; dm::sincos_(psi, sp, cp);
    vx = v * cp; vy = v * sp;
    x = x + vx * c.dt; y = y + vy * c.dt;
}
// rollout of a mother sample of mmd_opt: the 22 ridge-fit features (cem_helper.py:553-564, folded: feature_k = sum_t Wfit[k][t] * x[t],
// ascending t -- the contract's order) are accumulated while the state advances; the 22 independent fma chains fill the issue slots the
// serial sqrt -> tan -> sincos chain leaves empty.  Positions are written only for the kernels that still read them back (WRITE).
// MODE 0: features only; 1: also write the positions (kernels that read the mother rollouts back).  The latency regime does not come here: k_rollouts<ROLL_OPT>
// splits the rollout into its bare recurrence and parallel feature / maxima passes there.
template <int MODE>
__device__ __forceinline__ void rollout_fit(const DCfg& c, const float* a, const float* s, const float* st0, const float* __restrict__ W /* (11,np) */,
                                            float* __restrict__ xg, float* __restrict__ yg, float* __restrict__ feat) {
    float x = st0[0], y = st0[1], vx = st0[2], vy = st0[3], psi = st0[4];
    float fx[NV], fy[NV];
#pragma unroll
    for (int k = 0; k < NV; k++) { fx[k] = 0.0f; fy[k] = 0.0f; }
    const int np = c.np;
#pragma unroll 1
    for (int t = 0; t < np; t++) {          // the state BEFORE step t is the recorded point  [cem_helper.py:451-458]
        if (MODE == 1) { xg[t] = x; yg[t] = y; }
#pragma unroll
        for (int k = 0; k < NV; k++) { const float w = W[k * np + t]; fx[k] = fmaf(w, x, fx[k]); fy[k] = fmaf(w, y, fy[k]); }
        bicycle_step(c, a[t], s[t], x, y, vx, vy, psi);          // s = tan(steer), see k_rollouts
    }
#pragma unroll
    for (int k = 0; k < NV; k++) { feat[k] = fx[k]; feat[NV + k] = fy[k]; }
}
// MMD of nr scalar costs against the zero cost, kernel form KER (dm::KER_*)  [kernel_computation.py:67-87]
template <int KER = dm::KER_LAPLACE>
__device__ __noinline__ float mmd_cost(const DCfg& c, const float* beta, const float* cost, float sigma) {
    const int nr = c.nr;
    const float v = dm::kern_cost_v(KER, sigma);
    float s1 = 0.0f, s2 = 0.0f;
    for (int i = 0; i < nr; i++) {
        float t = 0.0f;
        for (int j = 0; j < nr; j++) t = fmaf(dm::kern_cost(KER, cost[i] - cost[j], v), beta[j], t);
        s1 = fmaf(beta[i], t, s1);
        float e = dm::kern_cost(KER, cost[i] - 0.0f, v), u = 0.0f;
        for (int j = 0; j < nr; j++) u = fmaf(e, c.beta_del, u);
        s2 = fmaf(beta[i], u, s2);
    }
    return c.ker_wt * (s1 - 2.0f * s2);
}
// the same value computed by a whole warp (num_reduced <= 64): lane l evaluates the kernel rows i = l, l + 32 as the same ascending-j
// fma chains, then every lane folds them in ascending i -- bit-identical to mmd_cost, nr^2 / 32 exps per lane instead of nr^2 on one.  Kernel form: c.kernel
__device__ __forceinline__ float mmd_cost_warp(const DCfg& c, const float* beta, const float* cost, float sigma, int lane) {
    const int nr = c.nr;
    const float v = dm::kern_cost_v(c.kernel, sigma);
    float tv[2] = {0.0f, 0.0f}, uv[2] = {0.0f, 0.0f};
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int i = lane + 32 * h;
        if (i < nr) {
            float t = 0.0f;
            for (int j = 0; j < nr; j++) t = fmaf(dm::kern_cost(c.kernel, cost[i] - cost[j], v), beta[j], t);
            const float e = dm::kern_cost(c.kernel, cost[i] - 0.0f, v);
            float u = 0.0f;
            for (int j = 0; j < nr; j++) u = fmaf(e, c.beta_del, u);
            tv[h] = t; uv[h] = u;
        }
    }
    float s1 = 0.0f, s2 = 0.0f;
    for (int i = 0; i < nr; i++) {
        const float t = __shfl_sync(FULL, i < 32 ? tv[0] : tv[1], i & 31), u = __shfl_sync(FULL, i < 32 ? uv[0] : uv[1], i & 31);
        s1 = fmaf(beta[i], t, s1);
        s2 = fmaf(beta[i], u, s2);
    }
    return c.ker_wt * (s1 - 2.0f * s2);
}
// CVaR of nr per-rollout costs: jnp.quantile (linear interpolation) + mean of the tail  [costs.py:213-220], by a whole warp (num_reduced <= 64): the two
// order statistics the quantile needs come from a stable RANK COUNT -- lane l ranks
// elements l and l + 32 against all nr values (O(nr) per lane instead of lane 0's O(nr^2) insertion sort), the lanes holding ranks floor(q) / ceil(q)
// broadcast their values -- and the tail mean keeps the contract's sequential ascending-index sum (nr adds on one lane): the value of a stable sort + scan, bit for bit.
__device__ __forceinline__ float cvar_cost_warp(const DCfg& c, const float* v, int lane) {
    const int nr = c.nr;
    const float q = c.alpha_quant * (float)(nr - 1);
    const float lo = floorf(q), hi = ceilf(q);
    const float hw = q - lo, lw = 1.0f - hw;
    int ilo = (int)lo, ihi = (int)hi;
    ilo = ilo < 0 ? 0 : (ilo > nr - 1 ? nr - 1 : ilo);
    ihi = ihi < 0 ? 0 : (ihi > nr - 1 ? nr - 1 : ihi);
    float vlo = 0.0f, vhi = 0.0f;
#pragma unroll
    for (int h = 0; h < 2; h++) {
        const int i = lane + 32 * h;
        const float vi = i < nr ? v[i] : 0.0f;
        int rank = -1;
        if (i < nr) {
            rank = 0;
            for (int j = 0; j < nr; j++) {
                const float vj = v[j];
                const bool less = dm::lt_nanlast(vj, vi), tie = !less && !dm::lt_nanlast(vi, vj);
                rank += (less || (tie && j < i)) ? 1 : 0;             // stable ascending order, NaN last
            }
        }
        const unsigned mlo = __ballot_sync(FULL, rank == ilo), mhi = __ballot_sync(FULL, rank == ihi);
        const float slo = __shfl_sync(FULL, vi, mlo ? __ffs(mlo) - 1 : 0), shi = __shfl_sync(FULL, vi, mhi ? __ffs(mhi) - 1 : 0);
        if (mlo) vlo = slo;
        if (mhi) vhi = shi;
    }
    const float var = vlo * lw + vhi * hw;
    float s = 0.0f; int n = 0;
    if (lane == 0) for (int i = 0; i < nr; i++) if (v[i] >= var) { s = s + v[i]; n++; }
    return n > 0 ? s / (float)n : 0.0f;          // valid on lane 0
}

// ---------------------------------------------------------------------------------------------
// k_rollouts: noisy controls + Euler rollouts, one thread per rollout.  Cost kinds with num_reduced rollouts (cvar / saa / mmd_random) finish
// here with their risk functional; mmd_opt writes the ridge-fit features of the num_reduced^2 mother rollouts (and the sample's noisy
// controls) for the inner-CEM kernel -- the rollouts themselves never leave the registers.  The solve is split into small kernels on
// purpose: v1 of this file, one fused kernel of 13.7k SASS instructions, spent 6.7 issue slots stalled on instruction fetch per instruction
// issued (profiles/r01_v1_summary.md), and every later measurement confirmed that code size is the first-order cost here
// (profiles/r01_v9_summary.md).
#define ROLL_THREADS 128
struct RollArgs {
    RiskArgs r;
    int spb;                 // samples per CTA
    int R;                   // rollouts per sample (nr or nr*nr)
    int stage_ctrl;          // cvar / saa / mmd_random: draw the noisy controls into shared memory with the whole CTA first (latency regime: few samples)
    int write_rolls;         // mmd_opt: also write the mother rollouts (only the generic / warp-per-chain inner kernels read them back)
    int fold_risk;           // mmd_opt, small launches: the mother rollouts also fold their obstacle / lane maxima into mrisk, k_opt_risk does not re-roll
    float* mrisk;            // [n][nm][3]
    float *xroll, *yroll;    // [n][R][np]   (mmd_opt, write_rolls only)
    float* feat;             // [n][nm][22]  (mmd_opt only)
    float* ctrl;             // [n][2][nr*np]  noisy acceleration and tan(noisy steering) of the sample (mmd_opt): k_opt_risk re-rolls the chosen reduced set from them
    float* stash;            // [persistent CTAs][S][32]  row stash of k_inner_cem_warp
    int* ridx;               // [n][nr]  reduced set chosen by k_inner_cem_fast, read by k_opt_risk
    float* bscratch;         // [n][S][nr + 1]  per-row beta vectors and packed reduced-set indices of k_inner_cem_fast's current iteration
};
// mmd_opt: noisy controls of the CTA's samples (2 x nr x np each) + the ridge-fit matrix; the other costs: 4 slots of per-rollout values
__host__ __device__ inline int roll_tail_floats(int nr) { return nr <= 16 ? 16 : ((nr + 3) & ~3); }
__host__ __device__ inline int roll_smem_floats(int spb, int nr, int np, int R, int stage_ctrl = 0, int fold = 0) {
    return R == nr ? spb * (4 * roll_tail_floats(nr) + (stage_ctrl ? 2 * nr * np : 0)) : spb * 2 * nr * np + ((NV * np + 3) & ~3) + (fold ? spb * R * 2 * np : 0);
}

// noisy control pair of element el = row * np + t of sample g  [cem_helper.py:405-443 / 470-508]
// NZ = the noise path the launch needs, fixed at compile time so that a kernel carries only that path's code and registers: 0 Gaussian, 1 Beta draws replayed from the
// per-episode candidate table (every beta-noise solve), 2 decided at run time (injected draws / direct sampler of the stage entry points)
enum { NZ_GAUSS = 0, NZ_BETA_TABLE = 1, NZ_ANY = 2 };
template <int NZ = NZ_ANY, bool PF = false>
__device__ __forceinline__ void noisy_control(const DCfg& c, const RiskArgs& a, int g, int e, int el, int t, int n, float& an, float& sn) {
    const float av = a.acc[(size_t)g * T_ + t], sv = a.steer[(size_t)g * T_ + t];
    const float* z3 = a.z3 + e * a.z_stride;
    float pa, ps;
    if (NZ == NZ_GAUSS || (NZ == NZ_ANY && c.noise_kind == 0)) {
        pa = (c.sigma_acc * fabsf(av)) * (a.z1 + e * a.z_stride)[el];
        ps = (c.sigma_steer * fabsf(sv)) * (a.z2 + e * a.z_stride)[el];
    } else {
        const uint32_t* keys = a.keys + e * a.key_stride;
        dr::Key k1, k2; k1.k0 = keys[0]; k1.k1 = keys[1]; k2.k0 = keys[2]; k2.k1 = keys[3];
        float b1, b2;
        if (NZ == NZ_ANY && a.binj1) {
            b1 = a.binj1[(size_t)g * n + el]; b2 = a.binj2[(size_t)g * n + el];
        } else if (NZ == NZ_BETA_TABLE || a.btab) {
            const float* bt = a.btab + e * a.btab_stride;
            b1 = dr::beta_replay<PF>(bt, k1, (uint32_t)n, (uint32_t)el, c.beta_a * fabsf(av), c.beta_b * fabsf(av));
            b2 = dr::beta_replay<PF>(bt + (size_t)2 * GT_FIELDS * n, k2, (uint32_t)n, (uint32_t)el, c.beta_a * fabsf(sv), c.beta_b * fabsf(sv));
        } else {
            b1 = dr::beta_elem(k1, (uint32_t)n, (uint32_t)el, c.beta_a * fabsf(av), c.beta_b * fabsf(av));
            b2 = dr::beta_elem(k2, (uint32_t)n, (uint32_t)el, c.beta_a * fabsf(sv), c.beta_b * fabsf(sv));
        }
        pa = c.sigma_acc * (2.0f * b1 - 1.0f);
        ps = c.ksig_steer * (2.0f * b2 - 1.0f);
    }
    an = (av + pa) + c.acc_const * z3[el];
    sn = (sv + ps) + c.steer_const * z3[el];
}

// Many obstacles (configs[4]: 32): the indicator of obstacle o at knot t is exactly 0 unless |x - xo| < a_obs (fbar's screen: A >= a^2 makes the rounded
// cost <= 0), so only the obstacles inside an x window around the vehicle can raise the maximum.  k_obs_sort orders every knot's obstacles by x once
// per solve; the rollout binary-searches the window (2-5 obstacles instead of 32).  Exact: the window is 0.01 m wider than a_obs (rounding of
// x +- w at |x| < 1e4 is < 5e-4), skipped obstacles contribute exactly 0, and the maximum is order independent; NaN positions (vehicle or
// obstacle) and |x| >= 1e4 take the plain loop, so NaN propagation is unchanged.
#define OBS_SORT_MIN 8
__global__ void k_obs_sort(const float* __restrict__ x_obs, const float* __restrict__ y_obs, float* __restrict__ sx, float* __restrict__ sy,
                           int* __restrict__ nan_flag, int O, int n_knots /* = n_ep * 100 */) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_knots) return;
    const int e = i / T_, t = i % T_;
    float xs[MPCMMD_MAX_NR_DEV], ys[MPCMMD_MAX_NR_DEV];
    int bad = 0;
    for (int o = 0; o < O; o++) {                     // stable insertion sort by x (NaN last)
        const float xv = x_obs[((size_t)e * O + o) * T_ + t], yv = y_obs[((size_t)e * O + o) * T_ + t];
        bad |= (xv != xv) || (yv != yv);
        int j = o;
        while (j > 0 && dm::lt_nanlast(xv, xs[j - 1])) { xs[j] = xs[j - 1]; ys[j] = ys[j - 1]; j--; }
        xs[j] = xv; ys[j] = yv;
    }
    for (int o = 0; o < O; o++) { sx[(size_t)i * O + o] = xs[o]; sy[(size_t)i * O + o] = ys[o]; }
    nan_flag[i] = bad;
}

// one rollout with its obstacle / lane indicators folded in: m = max over (obstacle, t) of f_bar, l / u = max over t of the lane violations,
// each evaluated on the state BEFORE step t (the recorded point).  The maxima are order independent (NaN propagates either way), so this equals
// the reference's "roll out, then reduce" [costs.py:50-71].  FLY: the controls of row `row` are drawn inside the loop (costs with one control row
// per rollout); otherwise they are read from a / s.
// SORTED = the launch has sorted obstacle windows (num_obs > OBS_SORT_MIN); a separate instantiation, so that the few-obstacle kernels do not carry the
// window search's code and registers (the combined kernel took k_rollouts<ROLL_FLY> from 341 to 549 us per 20 000-sample launch of configs[1])
template <bool FLY, bool SORTED = false, int NZ = NZ_ANY>
__device__ __forceinline__ void rollout_risk(const DCfg& c, const RiskArgs& A, int g, int e, int row, const float* a, const float* s,
                                             const float* st0, const float* __restrict__ xo, const float* __restrict__ yo, float& m, float& l, float& u) {
    float x = st0[0], y = st0[1], vx = st0[2], vy = st0[3], psi = st0[4];
    const int np = c.np, n = c.nr * np;
    m = 0.0f; l = 0.0f; u = 0.0f;
#pragma unroll 1
    for (int t = 0; t < np; t++) {
        float at, st;
        if (FLY) { noisy_control<NZ>(c, A, g, e, row * np + t, t, n, at, st); st = dm::tan_(st); } else { at = a[t]; st = s[t]; }      // s = tan(steer) when staged
        if (SORTED && A.sx_obs && x == x && y == y && fabsf(x) < 1.0e4f && !A.obs_nan[e * T_ + t]) {
            const float* xs = A.sx_obs + ((size_t)e * T_ + t) * c.O; const float* ys = A.sy_obs + ((size_t)e * T_ + t) * c.O;
            const float xl = x - c.obs_win, xh = x + c.obs_win;
            int lo = 0, n_ = c.O;
            while (n_ > 0) { const int half = n_ >> 1; if (xs[lo + half] <= xl) { lo += half + 1; n_ -= half + 1; } else n_ = half; }     // first obstacle with xs > x - w
#pragma unroll 1
            for (int i = lo; i < c.O; i++) {
                const float xv = xs[i];
                if (!(xv < xh)) break;
                m = dm::nmax_(m, fbar(c, x, y, xv, ys[i]));
            }
        } else {
#pragma unroll 4
            for (int o = 0; o < c.O; o++) m = dm::nmax_(m, fbar(c, x, y, xo[o * T_ + t], yo[o * T_ + t]));
        }
        l = dm::nmax_(l, dm::max0_(-y + c.y_lb));
        u = dm::nmax_(u, dm::max0_(y - c.y_ub));
        bicycle_step(c, at, st, x, y, vx, vy, psi);
    }
}

// MODE 0: mmd_opt; 1: num_reduced-rollout costs, throughput regime; 2: the same, latency regime.  Three instantiations keep each launch's code small.
enum { ROLL_OPT = 0, ROLL_FLY = 1, ROLL_STAGED = 2 };
// OV (ROLL_OPT only) = which of the three mmd_opt bodies the launch runs, fixed at compile time so that the throughput kernel does not carry the other two (the
// combined kernel was 4500 SASS instructions, instruction-fetch stalls 2.5 per issue): 0 features only, 1 also the mother rollouts' positions (generic / warp-per-chain
// inner kernels read them back), 2 the latency regime (RollArgs::fold_risk)
enum { OV_PLAIN = 0, OV_WRITE = 1, OV_FOLD = 2 };
template <int MODE, bool SORTED = false, int NZ = NZ_ANY, int OV = OV_PLAIN>
__global__ void __launch_bounds__(ROLL_THREADS) k_rollouts(DCfg c, RollArgs ra) {
    extern __shared__ __align__(128) float sm[];
    const RiskArgs& a = ra.r;
    const int tid = threadIdx.x, nt = ROLL_THREADS, warp = tid >> 5, lane = tid & 31;
    const int nr = c.nr, np = c.np, n = nr * np, R = ra.R, spb = ra.spb;
    const int g0 = blockIdx.x * spb;
    const int ns = min(spb, a.n_samples - g0);                 // samples in this CTA
    if (ns <= 0) return;
    if constexpr (MODE == ROLL_OPT) {
        // ================= mmd_opt: noisy controls -> num_reduced^2 mother rollouts -> ridge-fit features =================
        float* sW = sm + spb * 2 * n;
#pragma unroll 1
        for (int i = tid; i < NV * np; i += nt) sW[i] = c.Wfit[i];
#pragma unroll 1
        for (int i = tid; i < ns * n; i += nt) {
            const int ls = i / n, el = i % n, g = g0 + ls;
            float an, sn; noisy_control<NZ, OV == OV_FOLD>(c, a, g, g / a.B, el, el % np, n, an, sn);      // latency regime: prefetching replay
            const float tn = dm::tan_(sn);                     // the rollouts (and k_opt_risk's re-rolls) only ever need tan(steer)
            sm[ls * 2 * n + el] = an; sm[ls * 2 * n + n + el] = tn;
            ra.ctrl[(size_t)g * 2 * n + el] = an; ra.ctrl[(size_t)g * 2 * n + n + el] = tn;
        }
        __syncthreads();
        if constexpr (OV == OV_FOLD) {
            // ---- latency regime (a handful of samples per SM): the serial part of a mother rollout is reduced to the bare bicycle recurrence -- positions go to
            //      shared memory -- and everything that only READS the positions runs in parallel afterwards: one thread per (rollout, feature) for the 22
            //      ridge-fit chains (ascending t: the contract's order), one warp per rollout with a lane per knot for the obstacle / lane maxima.
            float* pos = sW + ((NV * np + 3) & ~3);                 // [ns][R][2][np]
#pragma unroll 1
            for (int i = tid; i < ns * R; i += nt) {
                const int ls = i / R, m = i % R, e = (g0 + ls) / a.B;
                const float* an = sm + ls * 2 * n + (m / nr) * np; const float* sn = sm + ls * 2 * n + n + (m % nr) * np;
                float* px = pos + (size_t)i * 2 * np; float* py = px + np;
                const float* st0 = a.state0 + e * 5;
                float x = st0[0], y = st0[1], vx = st0[2], vy = st0[3], psi = st0[4];
#pragma unroll 1
                for (int t = 0; t < np; t++) { px[t] = x; py[t] = y; bicycle_step(c, an[t], sn[t], x, y, vx, vy, psi); }
            }
            __syncthreads();
#pragma unroll 1
            for (int task = tid; task < ns * R * 2 * NV; task += nt) {
                const int i = task / (2 * NV), kk = task % (2 * NV), k = kk < NV ? kk : kk - NV;
                const float* p = pos + (size_t)i * 2 * np + (kk < NV ? 0 : np); const float* w = sW + k * np;
                float f = 0.0f;
#pragma unroll 5
                for (int t = 0; t < np; t++) f = fmaf(w[t], p[t], f);
                ra.feat[((size_t)g0 * R + i) * 2 * NV + kk] = f;
            }
#pragma unroll 1
            for (int i = warp; i < ns * R; i += nt / 32) {
                const int ls = i / R, e = (g0 + ls) / a.B;
                const float* px = pos + (size_t)i * 2 * np; const float* py = px + np;
                const float* xo = a.x_obs + (size_t)e * c.O * T_; const float* yo = a.y_obs + (size_t)e * c.O * T_;
                float m = 0.0f, l = 0.0f, u = 0.0f;
                for (int t = lane; t < np; t += 32) {
                    const float x = px[t], y = py[t];
#pragma unroll 4
                    for (int o = 0; o < c.O; o++) m = dm::nmax_(m, fbar(c, x, y, xo[o * T_ + t], yo[o * T_ + t]));
                    l = dm::nmax_(l, dm::max0_(-y + c.y_lb));
                    u = dm::nmax_(u, dm::max0_(y - c.y_ub));
                }
                m = warp_nmax(m); l = warp_nmax(l); u = warp_nmax(u);
                if (lane == 0) { float* mr = ra.mrisk + ((size_t)g0 * R + i) * 3; mr[0] = m; mr[1] = l; mr[2] = u; }
            }
            return;
        }
        // mother sample m = i*nr + j uses acc noise i, steer noise j  [cem_helper.py:510-511]
#pragma unroll 1
        for (int i = tid; i < ns * R; i += nt) {
            const int ls = i / R, m = i % R, g = g0 + ls, e = g / a.B;
            const float* an = sm + ls * 2 * n + (m / nr) * np; const float* sn = sm + ls * 2 * n + n + (m % nr) * np;
            float* ft = ra.feat + ((size_t)g * R + m) * 2 * NV;
            if constexpr (OV == OV_WRITE) rollout_fit<1>(c, an, sn, a.state0 + e * 5, sW, ra.xroll + ((size_t)g * R + m) * np, ra.yroll + ((size_t)g * R + m) * np, ft);
            else rollout_fit<0>(c, an, sn, a.state0 + e * 5, sW, nullptr, nullptr, ft);
        }
    } else {
    // ================= cvar / saa / mmd_random: one thread per (sample, rollout), controls drawn inside the rollout =================
    // Throughput regime: every thread draws its rollout's controls inside the loop (no staging, 25 samples per CTA).  Latency regime (a launch
    // too small to fill the GPU): the 2 x nr x np draws of a sample are spread over the whole CTA first, then nr threads roll out.
    const int tail = roll_tail_floats(nr), per = 4 * tail + (MODE == ROLL_STAGED ? 2 * n : 0);
    if constexpr (MODE == ROLL_STAGED) {
#pragma unroll 1
        for (int i = tid; i < ns * n; i += nt) {
            const int ls = i / n, el = i % n, g = g0 + ls;
            float an, sn; noisy_control<NZ, true>(c, a, g, g / a.B, el, el % np, n, an, sn);      // latency regime: prefetching replay
            sm[ls * per + 4 * tail + el] = an; sm[ls * per + 4 * tail + n + el] = dm::tan_(sn);
        }
        __syncthreads();
    }
    if constexpr (MODE == ROLL_STAGED) {
        // rollouts overwrite their own control rows in place (rollout r reads only row r), then one warp per sample reduces the obstacle / lane
        // indicators with a lane per timestep: the serial part of the CTA is just the np bicycle steps
#pragma unroll 1
        for (int i = tid; i < ns * R; i += nt) {
            const int ls = i / R, r = i % R, e = (g0 + ls) / a.B;
            float* an = sm + ls * per + 4 * tail + r * np; float* sn = an + n;
            float x = a.state0[e * 5], y = a.state0[e * 5 + 1], vx = a.state0[e * 5 + 2], vy = a.state0[e * 5 + 3], psi = a.state0[e * 5 + 4];
            for (int t = 0; t < np; t++) {
                const float at = an[t], st = sn[t];
                an[t] = x; sn[t] = y;
                bicycle_step(c, at, st, x, y, vx, vy, psi);
            }
        }
        __syncthreads();
#pragma unroll 1
        for (int ls = warp; ls < ns; ls += nt / 32) {
            const int e = (g0 + ls) / a.B;
            const float* xo = a.x_obs + (size_t)e * c.O * T_; const float* yo = a.y_obs + (size_t)e * c.O * T_;
            float* cst = sm + ls * per;
#pragma unroll 1
            for (int r = 0; r < nr; r++) {
                const float* xr = sm + ls * per + 4 * tail + r * np; const float* yr = xr + n;
                float m = 0.0f, l = 0.0f, u = 0.0f;
                for (int t = lane; t < np; t += 32) {
                    const float x = xr[t], y = yr[t];
#pragma unroll 4
                    for (int o = 0; o < c.O; o++) m = dm::nmax_(m, fbar(c, x, y, xo[o * T_ + t], yo[o * T_ + t]));
                    l = dm::nmax_(l, dm::max0_(-y + c.y_lb));
                    u = dm::nmax_(u, dm::max0_(y - c.y_ub));
                }
                m = warp_nmax(m); l = warp_nmax(l); u = warp_nmax(u);
                if (lane == 0) { cst[r] = m; cst[tail + r] = l; cst[2 * tail + r] = u; }
            }
        }
    } else {
#pragma unroll 1
        for (int i = tid; i < ns * R; i += nt) {
            const int ls = i / R, r = i % R, g = g0 + ls, e = g / a.B;
            float m, l, u;
            rollout_risk<true, SORTED, NZ>(c, a, g, e, r, nullptr, nullptr, a.state0 + e * 5, a.x_obs + (size_t)e * c.O * T_, a.y_obs + (size_t)e * c.O * T_, m, l, u);
            float* cst = sm + ls * per;
            cst[r] = m; cst[tail + r] = l; cst[2 * tail + r] = u;
        }
    }
    __syncthreads();
    // ---- risk functional of the nr per-rollout values (one warp per sample at a time)  [costs.py:137-234; cem.py:355-356]
#pragma unroll 1
    for (int ls = warp; ls < ns; ls += nt / 32) {
        const int g = g0 + ls;
        float* cst = sm + ls * per; float* lb = cst + tail; float* ub = lb + tail; float* bet = ub + tail;
        if (a.cost_kind == 1) {                           // mmd_random: beta = 1/nr, sigma = 0.01, lane = 0  [cem.py:355-356, 404-424]
            for (int i = lane; i < nr; i += 32) { bet[i] = c.beta_del; a.beta[(size_t)g * nr + i] = c.beta_del; }
            __syncwarp();
            const float risk = mmd_cost_warp(c, bet, cst, c.sigma_random, lane);
            if (lane == 0) { a.sigma[g] = c.sigma_random; a.risk[g] = risk; a.lane[g] = 0.0f; }
        } else if (a.cost_kind == 2) {                    // cvar  [costs.py:206-221, 137-158]: warp-level rank selection of the two quantile order statistics
            const float risk = cvar_cost_warp(c, cst, lane);
            const float lanec = cvar_cost_warp(c, lb, lane) + cvar_cost_warp(c, ub, lane);
            if (lane == 0) { a.risk[g] = risk; a.lane[g] = lanec; }
        } else if (lane == 0) {
            float risk, lanec;
            {                                             // saa  [costs.py:223-234, 160-171]
                float s = 0.0f, sl = 0.0f, su = 0.0f;
                for (int i = 0; i < nr; i++) { s = s + (cst[i] > 0.0f ? 1.0f : 0.0f); sl = sl + (lb[i] > 0.0f ? 1.0f : 0.0f); su = su + (ub[i] > 0.0f ? 1.0f : 0.0f); }
                risk = s / (float)nr;
                lanec = (sl + su) / (float)nr;
            }
            a.risk[g] = risk; a.lane[g] = lanec;
        }
    }
    }
}

// ---------------------------------------------------------------------------------------------
// k_inner_cem (mmd_opt): one CTA (3 warps) per sample: distance table, the reduced-set CEM, MMD risk of the chosen set.
// 89 = S - n_elite new beta samples are evaluated per inner iteration (the 11 elites keep last iteration's cost: same
// row => same arithmetic => same bits), so 96 threads are ~93 % busy in the sample stage and in the row-per-thread
// resampling stage.
#define RISKO_THREADS 96
#define RISKO_THREADS_BIG 512  // num_reduced^2 + 1 > 32: one CTA per SM (100+ KB of shared memory), so the CTA itself has to fill the SM
// measured per solve at 8 episodes (tools/time_generic_nr.py), 256 / 512 threads: num_reduced 6: 4.0 / 6.5 ms, 8: 13.4 / 11.9 ms, 10: 24.2 / 21.5 ms
__host__ __device__ constexpr int risko_threads(int nr) { return nr * nr + 1 <= 32 ? RISKO_THREADS : (nr <= 7 ? 256 : RISKO_THREADS_BIG); }

struct OptLayout {          // shared-memory carve-up (in floats); every offset is a multiple of 4 floats (16 B)
    int F, D, small, red, th, cost, betas, idxs, key64, perm, C, rd, mean, eth, xc, ecost, ebetas, eidxs, rs;
    int ldc, total;
};
__host__ __device__ inline int al4(int x) { return (x + 3) & ~3; }
__host__ __device__ inline OptLayout opt_layout(int nr, int np, int S, int ne) {
    OptLayout L; const int nm = nr * nr, d = nm + 1;
    (void)np;
    L.ldc = al4(d);
    int q = 0;
    L.F = q; q += al4(nm * 2 * NV); L.D = q; q += al4(nm * nm); L.small = q; q += 64;
    L.red = q; q += al4(3 * 16 * (RISKO_THREADS_BIG / 32));
    L.th = q; q += al4(S * d); L.cost = q; q += al4(S); L.betas = q; q += al4(S * nr); L.idxs = q; q += al4(S * nr);
    L.key64 = q; q += al4(2 * S); L.perm = q; q += al4(S); L.C = q; q += al4(d * L.ldc); L.rd = q; q += al4(d); L.mean = q; q += al4(d);
    L.eth = q; q += al4(ne * d); L.xc = q; q += al4(ne * d); L.ecost = q; q += al4(ne); L.ebetas = q; q += al4(ne * nr); L.eidxs = q; q += al4(ne * nr);
    L.rs = q; if (d > 32) q += al4(S * nr);           // per-(sample, reduced index) kernel row sums of the phased evaluation (large reduced sets)
    L.total = q;
    return L;
}

// one beta sample of the inner CEM: choose the top-NR |theta| (stable, ascending), build the Laplace kernels from the
// chain's distance table, solve the equality-constrained QP by Cholesky block elimination, return the MMD cost
// [compute_beta.py:113-129, 70-91].  |theta| is compared through its bit pattern (non-negative floats order like
// integers and NaN patterns sort last), which is the jnp.argsort order.
// the three stages of one beta sample; beta_sample = beta_topk -> beta_rowsum (x NR) -> beta_finish.  The generic kernel for large reduced
// sets runs them as separate block-wide phases (one task per (sample, reduced index) in the exp-heavy middle stage).
template <int NR>
__device__ __forceinline__ void beta_topk(const float* __restrict__ row, int* __restrict__ ti_out) {
    constexpr int nm = NR * NR;
    int tv[NR], ti[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) { tv[i] = -1; ti[i] = -1; }
#pragma unroll 1
    for (int m = 0; m < nm; m++) {                 // branch-free insertion: replace the smallest, bubble it up past <= elements
        const int v = (int)(dm::f2u(row[m]) & 0x7fffffffu);
        bool mv = v >= tv[0];
        tv[0] = mv ? v : tv[0]; ti[0] = mv ? m : ti[0];
#pragma unroll
        for (int p = 0; p < NR - 1; p++) {
            mv = mv && (tv[p] >= tv[p + 1]);
            const int a0 = tv[p], a1 = tv[p + 1], b0 = ti[p], b1 = ti[p + 1];
            tv[p] = mv ? a1 : a0; tv[p + 1] = mv ? a0 : a1; ti[p] = mv ? b1 : b0; ti[p + 1] = mv ? b0 : b1;
        }
    }
#pragma unroll
    for (int i = 0; i < NR; i++) ti_out[i] = ti[i];
}
// sum_m k(D[m][ti]; sigma), ascending m  [kernel_computation.py:31-37, compute_beta.py:77]; D is symmetric bit for bit
template <int KER = dm::KER_LAPLACE>
__device__ __forceinline__ float beta_rowsum(const float* __restrict__ D, int nm, int ti, float sigma) {
    const dm::LapScale ls = dm::kern_scale<KER>(sigma);
    float acc = 0.0f;
#pragma unroll 4
    for (int m = 0; m < nm; m++) acc = acc + dm::lap_(D[m * nm + ti], ls);
    return acc;
}
template <int NR, int KER = dm::KER_LAPLACE>
__device__ __forceinline__ float beta_finish(const DCfg& c, const int* __restrict__ ti, float sigma, const float* __restrict__ rowsum,
                                             const float* __restrict__ D, float* __restrict__ beta_out) {
    constexpr int nm = NR * NR;
    const dm::LapScale ls = dm::kern_scale<KER>(sigma);
    float K[NR][NR];                               // ker_red (symmetric bit for bit); diagonal: k(0) = 1
#pragma unroll
    for (int i = 0; i < NR; i++) {
        K[i][i] = 1.0f;
#pragma unroll
        for (int j = 0; j < i; j++) { const float k = dm::lap_(D[ti[i] * nm + ti[j]], ls); K[i][j] = k; K[j][i] = k; }
    }
    // A = ker_red + 0.05 I, Cholesky with reciprocal pivots
    float Lm[NR][NR], rd[NR], u[NR], w[NR];
#pragma unroll
    for (int j = 0; j < NR; j++) {
        float acc = K[j][j] + 0.05f;
#pragma unroll
        for (int k = 0; k < j; k++) acc = fmaf(-Lm[j][k], Lm[j][k], acc);
        const float dd = sqrtf(acc);
        Lm[j][j] = dd; rd[j] = 1.0f / dd;
#pragma unroll
        for (int i = j + 1; i < NR; i++) {
            float aa = K[i][j];
#pragma unroll
            for (int k = 0; k < j; k++) aa = fmaf(-Lm[i][k], Lm[j][k], aa);
            Lm[i][j] = aa * rd[j];
        }
    }
#pragma unroll
    for (int i = 0; i < NR; i++) {
        float aa = c.inv_nm * rowsum[i], bb = 1.0f;
#pragma unroll
        for (int k = 0; k < i; k++) { aa = fmaf(-Lm[i][k], u[k], aa); bb = fmaf(-Lm[i][k], w[k], bb); }
        u[i] = aa * rd[i]; w[i] = bb * rd[i];
    }
#pragma unroll
    for (int i = NR - 1; i >= 0; i--) {
        float aa = u[i], bb = w[i];
#pragma unroll
        for (int k = i + 1; k < NR; k++) { aa = fmaf(-Lm[k][i], u[k], aa); bb = fmaf(-Lm[k][i], w[k], bb); }
        u[i] = aa * rd[i]; w[i] = bb * rd[i];
    }
    float su = 0.0f, sw = 0.0f;
#pragma unroll
    for (int i = 0; i < NR; i++) { su = su + u[i]; sw = sw + w[i]; }
    const float nu = (su - 1.0f) / sw;
    float beta[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) beta[i] = fmaf(-nu, w[i], u[i]);
    float s1 = 0.0f, s2 = 0.0f;
#pragma unroll
    for (int i = 0; i < NR; i++) {
        float t = 0.0f;
#pragma unroll
        for (int j = 0; j < NR; j++) t = fmaf(K[i][j], beta[j], t);
        s1 = fmaf(beta[i], t, s1);
        s2 = fmaf(c.m2_inv_nm * rowsum[i], beta[i], s2);
    }
#pragma unroll
    for (int i = 0; i < NR; i++) beta_out[i] = beta[i];
    return s1 + s2;
}

template <int NR, int KER = dm::KER_LAPLACE>
__device__ __forceinline__ float beta_sample(const DCfg& c, const float* __restrict__ row, const float* __restrict__ D,
                                             float* __restrict__ beta_out, int* __restrict__ idx_out) {
    constexpr int nm = NR * NR;
    int ti[NR];
    beta_topk<NR>(row, ti);
    const float sigma = row[nm];
    const dm::LapScale ls = dm::kern_scale<KER>(sigma);
    float rowsum[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) rowsum[i] = 0.0f;
#pragma unroll 1
    for (int m = 0; m < nm; m++) {                 // D is symmetric bit for bit: read column m (bank-conflict free across threads)
        const float* Dm = D + m * nm;
#pragma unroll
        for (int i = 0; i < NR; i++) rowsum[i] = rowsum[i] + dm::lap_(Dm[ti[i]], ls);
    }
#pragma unroll
    for (int i = 0; i < NR; i++) idx_out[i] = ti[i];
    return beta_finish<NR, KER>(c, ti, sigma, rowsum, D, beta_out);
}

// float -> int64 key whose signed order is "ascending float, -0 == +0, NaN last", tie-broken by the index in the low bits
__device__ __forceinline__ long long sort_key64(float x, int idx) {
    const float xz = x + 0.0f;                                   // -0 -> +0
    const uint32_t ubits = dm::f2u(xz);
    int k = (ubits & 0x80000000u) ? (int)(~ubits ^ 0x80000000u) : (int)ubits;
    if (xz != xz) k = 0x7fffffff;
    return ((long long)k << 12) | (long long)idx;
}

// SC / NEC: compile-time copies of the inner CEM's sample / elite counts (0 = from the configuration), as in k_inner_cem_fast: the shared-memory layout folds
// KER: MMD kernel form (dm::KER_*)
template <int NR, int SC = 0, int NEC = 0, int KER = dm::KER_LAPLACE>
__global__ void __launch_bounds__(risko_threads(NR), (NR <= 5) ? 7 : 1) k_inner_cem(DCfg c, RollArgs ra) {
    extern __shared__ __align__(128) float sm[];
    const RiskArgs& a = ra.r;
    const int g = blockIdx.x;
    if (g >= a.n_samples) return;
    constexpr int nm = NR * NR, d = nm + 1;
    constexpr bool SMALL = d <= 32;
    constexpr int nt = risko_threads(NR);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int e = g / a.B, np = c.np, S = SC ? SC : c.S_in, ne = NEC ? NEC : c.n_el_in;
    const OptLayout L = opt_layout(NR, np, S, ne);
    const int ldc = L.ldc;
    float* F = sm + L.F; float* D = sm + L.D; float* small = sm + L.small;
    // ---- distance table of the mother features  [kernel_computation.py:31-33]
    {
        const float* Fg = ra.feat + (size_t)g * nm * 2 * NV;
#pragma unroll 1
        for (int i = tid; i < nm * 2 * NV; i += nt) F[i] = Fg[i];
    }
    __syncthreads();
#pragma unroll 1
    for (int i = tid; i < nm * nm; i += nt) {
        const float* Fa = F + (i / nm) * 2 * NV; const float* Fb = F + (i % nm) * 2 * NV;
        float dist = 0.0f;
#pragma unroll
        for (int f = 0; f < 2 * NV; f++) dist = dm::kern_dist_acc<KER>(dist, Fa[f], Fb[f]);
        D[i] = dist;
    }
    // ---- inner CEM  [compute_beta.py:93-157]
    float* th = sm + L.th; float* cost = sm + L.cost; float* betas = sm + L.betas; int* idxs = (int*)(sm + L.idxs);
    long long* key64 = (long long*)(sm + L.key64); int* perm = (int*)(sm + L.perm);
    float* C = sm + L.C; float* mean = sm + L.mean; float* eth = sm + L.eth; float* xc = sm + L.xc;
    float* ecost = sm + L.ecost; float* ebetas = sm + L.ebetas; int* eidxs = (int*)(sm + L.eidxs);
#pragma unroll 1
    for (int i = tid; i < S * d; i += nt) th[i] = __ldg(c.theta0 + i);
    __syncthreads();
    float* resb = a.res_beta + (size_t)g * c.iters_in;
#pragma unroll 1
    for (int it = 0; it < c.iters_in; it++) {
        // -- evaluate the new samples (all of them in iteration 0; afterwards rows 0..ne-1 are last iteration's elites)
        if constexpr (SMALL) {
#pragma unroll 1
            for (int s = (it == 0 ? 0 : ne) + tid; s < S; s += nt) cost[s] = beta_sample<NR, KER>(c, th + s * d, D, betas + s * NR, idxs + s * NR);
        } else {
            // phased evaluation: (A) top-NR per sample, (B) one task per (sample, reduced index): the nm-term kernel row sum -- 97 % of the
            // exponentials, spread over all threads instead of one thread per sample --, (C) the (nr+1) KKT solve and the cost per sample
            const int s0 = (it == 0 ? 0 : ne);
            float* rs = sm + L.rs;
#pragma unroll 1
            for (int s = s0 + tid; s < S; s += nt) beta_topk<NR>(th + s * d, idxs + s * NR);
            __syncthreads();
#pragma unroll 1
            for (int task = tid; task < (S - s0) * NR; task += nt) {
                const int s = s0 + task / NR, i = task % NR;
                rs[s * NR + i] = beta_rowsum<KER>(D, nm, idxs[s * NR + i], th[s * d + nm]);
            }
            __syncthreads();
#pragma unroll 1
            for (int s = s0 + tid; s < S; s += nt) cost[s] = beta_finish<NR, KER>(c, idxs + s * NR, th[s * d + nm], rs + s * NR, D, betas + s * NR);
        }
        __syncthreads();
#pragma unroll 1
        for (int s = tid; s < S; s += nt) key64[s] = sort_key64(cost[s], s);
        __syncthreads();
#pragma unroll 1
        for (int s = tid; s < S; s += nt) {        // stable argsort by rank counting; only the ne best are needed
            const long long ks = key64[s];
            int rank = 0;
#pragma unroll 4
            for (int j = 0; j < S; j++) rank += (key64[j] < ks) ? 1 : 0;
            if (rank < ne) perm[rank] = s;
        }
        __syncthreads();
        // -- gather the elites (rank order) and their mean  [compute_beta.py:56-60]
#pragma unroll 1
        for (int i = tid; i < ne * d; i += nt) eth[i] = th[perm[i / d] * d + (i % d)];
#pragma unroll 1
        for (int i = tid; i < ne * NR; i += nt) { const int src = perm[i / NR] * NR + (i % NR); ebetas[i] = betas[src]; eidxs[i] = idxs[src]; }
#pragma unroll 1
        for (int i = tid; i < ne; i += nt) ecost[i] = cost[perm[i]];
#pragma unroll 1
        for (int i = tid; i < d; i += nt) {
            float s = 0.0f;
            for (int el = 0; el < ne; el++) s = s + th[perm[el] * d + i];
            mean[i] = s / (float)ne;
        }
        __syncthreads();
#pragma unroll 1
        for (int i = tid; i < ne * d; i += nt) { const float v = eth[i]; th[i] = v; xc[i] = v - mean[i % d]; }
#pragma unroll 1
        for (int i = tid; i < ne * NR; i += nt) { betas[i] = ebetas[i]; idxs[i] = eidxs[i]; }
#pragma unroll 1
        for (int i = tid; i < ne; i += nt) cost[i] = ecost[i];
        __syncthreads();
#pragma unroll 1
        for (int i = tid; i < d * d; i += nt) {    // jnp.cov (ddof = 1) + 0.05 I, lower triangle  [compute_beta.py:61]
            const int r = i / d, q = i % d;
            if (q <= r) {
                float acc = 0.0f;
                for (int el = 0; el < ne; el++) acc = fmaf(xc[el * d + r], xc[el * d + q], acc);
                acc = acc / (float)(ne - 1);
                if (r == q) acc = acc + 0.05f;
                C[r * ldc + q] = acc;
            }
        }
        __syncthreads();
        if constexpr (SMALL) {
            // -- Cholesky by warp 0, one row per lane, left-looking: acc = a_ij - sum_k<j L_ik L_jk as an ascending-k fma chain
            if (warp == 0) {
#pragma unroll 1
                for (int j = 0; j < d; j++) {
                    float acc = 0.0f;
                    if (lane >= j && lane < d) {
                        acc = C[lane * ldc + j];
                        for (int k = 0; k < j; k++) acc = fmaf(-C[lane * ldc + k], C[j * ldc + k], acc);
                    }
                    const float ajj = __shfl_sync(FULL, acc, j);
                    const float dd = sqrtf(ajj);
                    const float rdj = 1.0f / dd;
                    if (lane == j) C[j * ldc + j] = dd;
                    else if (lane > j && lane < d) C[lane * ldc + j] = acc * rdj;
                    __syncwarp();
                }
            }
            __syncthreads();
            // -- resample: one thread per new row, normals in registers, L broadcast from shared memory  [compute_beta.py:63-66]
            const int nrow = S - ne;
            const float* zT = c.zb_iterT + (size_t)it * d * nrow;
#pragma unroll 1
            for (int r = tid; r < nrow; r += nt) {
                float z[d];
#pragma unroll
                for (int k = 0; k < d; k++) z[k] = __ldg(zT + k * nrow + r);
                float* dst = th + (ne + r) * d;
#pragma unroll
                for (int q = 0; q < d; q++) {
                    const float4* Cq = reinterpret_cast<const float4*>(C + q * ldc);
                    float acc = 0.0f;
#pragma unroll
                    for (int k4 = 0; k4 <= q / 4; k4++) {
                        const float4 l = Cq[k4];
                        if (4 * k4 + 0 <= q) acc = fmaf(l.x, z[4 * k4 + 0], acc);
                        if (4 * k4 + 1 <= q) acc = fmaf(l.y, z[4 * k4 + 1], acc);
                        if (4 * k4 + 2 <= q) acc = fmaf(l.z, z[4 * k4 + 2], acc);
                        if (4 * k4 + 3 <= q) acc = fmaf(l.w, z[4 * k4 + 3], acc);
                    }
                    float v = mean[q] + acc;
                    if (q == nm) v = (v != v) ? v : (v > c.sigma_clip ? v : c.sigma_clip);
                    dst[q] = v;
                }
            }
        } else {
            // -- block-wide Cholesky, left-looking by PANELS of four columns (same scheme as icf_chol_panel of k_inner_cem.cuh, one row per
            //    thread): four independent fma chains per thread over the finished columns k < j0, the 4 x 4 diagonal block published through
            //    shared memory and factored redundantly by every thread, the factor kept transposed in the upper triangle (LT[k][q] = L[q][k])
            //    where the resampling reads it.  2 block barriers per panel (52 for d = 101) instead of 2 per column (202), and no thread walks
            //    a single dependent chain.  Entry (r, j) still accumulates fma(-L_rk, L_jk, .) for k ascending, then sqrt / reciprocal scaling.
            float* blk = sm + L.rd;                            // 16 floats: diagonal-block partials b(u', u) at blk[4 u' + u]
            const int r = tid;
#pragma unroll 1
            for (int p = 0; p < (d + 3) / 4; p++) {
                const int j0 = 4 * p;
                const bool act = r < d && r >= j0;
                float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
                if (act) {
                    const float4 av = *reinterpret_cast<const float4*>(C + r * ldc + j0);
                    a0 = av.x; a1 = av.y; a2 = av.z; a3 = av.w;
#pragma unroll 4
                    for (int k = 0; k < j0; k++) {
                        const float lr = C[k * ldc + r];
                        const float4 lj = *reinterpret_cast<const float4*>(C + k * ldc + j0);
                        a0 = fmaf(-lr, lj.x, a0); a1 = fmaf(-lr, lj.y, a1); a2 = fmaf(-lr, lj.z, a2); a3 = fmaf(-lr, lj.w, a3);
                    }
                    if (r < j0 + 4) { float* b = blk + 4 * (r - j0); b[0] = a0; b[1] = a1; b[2] = a2; b[3] = a3; }
                }
                __syncthreads();
                if (act) {
                    const float b00 = blk[0], b10 = blk[4], b11 = blk[5], b20 = blk[8], b21 = blk[9], b22 = blk[10];
                    const float b30 = blk[12], b31 = blk[13], b32 = blk[14], b33 = blk[15];
                    const float d0 = sqrtf(b00), r0 = 1.0f / d0;
                    const float l10 = b10 * r0, l20 = b20 * r0, l30 = b30 * r0;
                    const float d1 = sqrtf(fmaf(-l10, l10, b11)), r1 = 1.0f / d1;
                    const float l21 = fmaf(-l20, l10, b21) * r1, l31 = fmaf(-l30, l10, b31) * r1;
                    const float d2 = sqrtf(fmaf(-l21, l21, fmaf(-l20, l20, b22))), r2 = 1.0f / d2;
                    const float l32 = fmaf(-l31, l21, fmaf(-l30, l20, b32)) * r2;
                    const float d3 = sqrtf(fmaf(-l32, l32, fmaf(-l31, l31, fmaf(-l30, l30, b33)))), r3 = 1.0f / d3;
                    float e0 = a0 * r0;
                    a1 = fmaf(-e0, l10, a1); float e1 = a1 * r1;
                    a2 = fmaf(-e1, l21, fmaf(-e0, l20, a2)); float e2 = a2 * r2;
                    a3 = fmaf(-e2, l32, fmaf(-e1, l31, fmaf(-e0, l30, a3))); float e3 = a3 * r3;
                    if (r == j0) e0 = d0;
                    if (r == j0 + 1) e1 = d1;
                    if (r == j0 + 2) e2 = d2;
                    if (r == j0 + 3) e3 = d3;
                    // column r of LT rows j0..j0+3 (q = r >= k only); the consumed sub-diagonal entries of row r are left as they are:
                    // the resampling below never reads the lower triangle
                    if (r >= j0 + 0) C[(j0 + 0) * ldc + r] = e0;
                    if (r >= j0 + 1 && j0 + 1 < d) C[(j0 + 1) * ldc + r] = e1;
                    if (r >= j0 + 2 && j0 + 2 < d) C[(j0 + 2) * ldc + r] = e2;
                    if (r >= j0 + 3 && j0 + 3 < d) C[(j0 + 3) * ldc + r] = e3;
                }
                __syncthreads();
            }
            // -- resample  [compute_beta.py:63-66]: task = (new row r, 8 consecutive columns q0..q0+7); acc_u = sum_{k <= q0+u} L[q0+u][k] z[r][k],
            //    k ascending (the contract's chain), with the 8 columns of a step read as two float4 of row k.  Warps take consecutive r for one
            //    column group: the L reads broadcast and the normals (a constant table, [iter][k][row]) are read coalesced from L1/L2.
            const int nrow = S - ne;
            const float* zT = c.zb_iterT + (size_t)it * d * nrow;
            constexpr int NQ8 = (d + 7) / 8;
#pragma unroll 1
            for (int task = tid; task < NQ8 * nrow; task += nt) {
                const int q0 = 8 * (task / nrow), r = task % nrow;
                float acc[8];
#pragma unroll
                for (int u = 0; u < 8; u++) acc[u] = 0.0f;
                const float* zp = zT + r;
#pragma unroll 2
                for (int k = 0; k <= q0; k++) {                 // every column of the group has q >= k
                    const float z = __ldg(zp + (size_t)k * nrow);
                    const float4 l0 = *reinterpret_cast<const float4*>(C + k * ldc + q0), l1 = *reinterpret_cast<const float4*>(C + k * ldc + q0 + 4);
                    acc[0] = fmaf(l0.x, z, acc[0]); acc[1] = fmaf(l0.y, z, acc[1]); acc[2] = fmaf(l0.z, z, acc[2]); acc[3] = fmaf(l0.w, z, acc[3]);
                    acc[4] = fmaf(l1.x, z, acc[4]); acc[5] = fmaf(l1.y, z, acc[5]); acc[6] = fmaf(l1.z, z, acc[6]); acc[7] = fmaf(l1.w, z, acc[7]);
                }
#pragma unroll
                for (int kk = 1; kk < 8; kk++) {                // the triangle inside the group: column q0+u takes k = q0+kk only if u >= kk
                    const int k = q0 + kk;
                    if (k < d) {
                        const float z = __ldg(zp + (size_t)k * nrow);
#pragma unroll
                        for (int u = kk; u < 8; u++) if (q0 + u < d) acc[u] = fmaf(C[k * ldc + q0 + u], z, acc[u]);
                    }
                }
                float* dst = th + (ne + r) * d + q0;
#pragma unroll
                for (int u = 0; u < 8; u++) {
                    if (q0 + u < d) {
                        float v = mean[q0 + u] + acc[u];
                        if (q0 + u == nm) v = (v != v) ? v : (v > c.sigma_clip ? v : c.sigma_clip);
                        dst[u] = v;
                    }
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            resb[it] = ecost[0];
            if (it == c.iters_in - 1) {            // beta / reduced set of the best sample; sigma from the RESAMPLED array [Q7]
                for (int i = 0; i < NR; i++) { small[i] = ebetas[i]; ((int*)small)[16 + i] = eidxs[i]; }
                small[48] = th[perm[0] * d + nm];
            }
        }
        __syncthreads();
    }
    // ---- risk of the chosen reduced set (its rollouts come back from global memory)  [costs.py:173-186, 121-135]
    const int* ridx = (const int*)small + 16;
    const float* xg = ra.xroll + (size_t)g * nm * np; const float* yg = ra.yroll + (size_t)g * nm * np;
    const float* xo = a.x_obs + (size_t)e * c.O * T_; const float* yo = a.y_obs + (size_t)e * c.O * T_;
    constexpr int NW = nt / 32;
    float* red = sm + L.red;  // per-warp partial maxima, 3 * NR * NW floats
#pragma unroll 1
    for (int r = 0; r < NR; r++) {
        const float* xred = xg + ridx[r] * np; const float* yred = yg + ridx[r] * np;
        float m = 0.0f, l = 0.0f, u = 0.0f;
        for (int i = tid; i < c.O * np; i += nt) {
            const int o = i / np, t = i % np;
            m = dm::nmax_(m, fbar(c, xred[t], yred[t], xo[o * T_ + t], yo[o * T_ + t]));
        }
        for (int t = tid; t < np; t += nt) {
            l = dm::nmax_(l, dm::max0_(-yred[t] + c.y_lb));
            u = dm::nmax_(u, dm::max0_(yred[t] - c.y_ub));
        }
        m = warp_nmax(m); l = warp_nmax(l); u = warp_nmax(u);
        if (lane == 0) { red[(r * 3 + 0) * NW + warp] = m; red[(r * 3 + 1) * NW + warp] = l; red[(r * 3 + 2) * NW + warp] = u; }
    }
    __syncthreads();
    if (tid == 0) {
        float cs[NR], lbv[NR], ubv[NR], beta[NR];
        for (int r = 0; r < NR; r++) {
            float m = red[(r * 3 + 0) * NW], l = red[(r * 3 + 1) * NW], u = red[(r * 3 + 2) * NW];
            for (int wv = 1; wv < NW; wv++) { m = dm::nmax_(m, red[(r * 3 + 0) * NW + wv]); l = dm::nmax_(l, red[(r * 3 + 1) * NW + wv]); u = dm::nmax_(u, red[(r * 3 + 2) * NW + wv]); }
            cs[r] = m; lbv[r] = l; ubv[r] = u; beta[r] = small[r];
            a.beta[(size_t)g * NR + r] = small[r];
        }
        const float sigma = small[48];
        a.sigma[g] = sigma;
        a.risk[g] = mmd_cost<KER>(c, beta, cs, sigma);
        a.lane[g] = mmd_cost<KER>(c, beta, lbv, sigma) + mmd_cost<KER>(c, beta, ubv, sigma);
    }
}
