/*
 * include/mpcmmd.h -- C ABI of libmpcmmd.so, the B200 (sm_100a) implementation of the MPC-MMD
 * trajectory-optimizer inner loop.  Plain pointers and sizes only; no torch / C++ types.
 *
 * The reference (Basant1861/MPC-MMD) is pure Python on JAX: there is no FFI in it to re-bind.  The
 * interface this ABI replaces is the Python method surface of class CEM:
 *     CEM.__init__                       synthetic_static_obs/optimizer/cem.py:16-199   -> mpcmmd_create
 *     CEM.compute_cem_mmd_opt            synthetic_static_obs/optimizer/cem.py:201-333  -> mpcmmd_solve(kind 0)
 *     CEM.compute_cem_mmd_random         synthetic_static_obs/optimizer/cem.py:335-462  -> mpcmmd_solve(kind 1)
 *     CEM.compute_cem_cvar               synthetic_static_obs/optimizer/cem.py:464-588  -> mpcmmd_solve(kind 2)
 *     CEM.compute_cem_saa                synthetic_static_obs/optimizer/cem.py:590-714  -> mpcmmd_solve(kind 3)
 * called from synthetic_static_obs/main_mpc.py:113-119 (and synthetic_dynamic_obs/main_mpc.py:128-135).
 * One mpcmmd_solve call runs n_ep independent solves (the reference's per-episode loop,
 * main_mpc.py:106) in one batch.  INTEGRATION.md shows the ctypes binding that sits behind the
 * drop-in `optimizer.cem.CEM` class.
 *
 * Conventions: every function returns 0 on success, <0 on error (mpcmmd_last_error() gives the
 * text).  A handle serialises its work on the stream passed to each call.  "dev" pointers are
 * device pointers on the handle's device; "host" pointers are ordinary host memory.
 */
#ifndef MPCMMD_H
#define MPCMMD_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define MPCMMD_T 100      /* num   (cem.py:38)  knots per trajectory   */
#define MPCMMD_NVAR 11    /* nvar  (cem.py:50)  Bernstein coefficients */
#define MPCMMD_NPARAM 8   /* num_params (cem.py:136) */
#define MPCMMD_MAX_NR 10  /* largest num_reduced of the mmd_opt reduced-set kernels with shared-memory chain state */
#define MPCMMD_MAX_NR_OPT 40  /* largest num_reduced of mmd_opt (11..40: chain state in global memory, k_inner_cem_big) */
#define MPCMMD_MAX_NR_WIDE 1024  /* largest num_reduced of cvar / saa / mmd_random (2..64: warp-wide risk per sample; 65..1024: one CTA per sample, k_rollouts_wide) */

enum { MPCMMD_COST_MMD_OPT = 0, MPCMMD_COST_MMD_RANDOM = 1, MPCMMD_COST_CVAR = 2, MPCMMD_COST_SAA = 3 };
enum { MPCMMD_NOISE_GAUSSIAN = 0, MPCMMD_NOISE_BETA = 1 };
/* kernel of the MMD risk costs (mmd_opt, mmd_random): Laplace exp(-|d|_1 / sigma) as the reference, or Gaussian exp(-|d|_2^2 / (2 sigma^2)).
 * DESIGN.md section 3 items 4 and 8 fix the float32 arithmetic of both. */
enum { MPCMMD_KERNEL_LAPLACE = 0, MPCMMD_KERNEL_GAUSSIAN = 1 };

/* Every constant of CEM.__init__ (cem.py:20-171) the hot path reads.  The matrices are HOST
 * pointers, copied to the device by mpcmmd_create; the host shim computes them once in float64
 * (the folded constant solves of cem_helper.py:216-223, projection.py:145-168, cem_helper.py:553-564). */
typedef struct {
    int32_t num_batch;          /* cem.py:137 (100) */
    int32_t num_prime;          /* cem.py:52 */
    int32_t num_reduced;        /* cem.py:142 */
    int32_t num_obs;
    int32_t maxiter_cem;        /* cem.py:89 (20) */
    int32_t ellite_num;         /* cem.py:138 (5) */
    int32_t ellite_num_cost;    /* cem.py:140 (20) */
    int32_t noise_kind;         /* MPCMMD_NOISE_* (cem_helper.py:405/416) */
    int32_t num_samples_cem;    /* compute_beta.py:14 (100) */
    int32_t maxiter_beta_cem;   /* compute_beta.py:15 (20) */
    int32_t num_ellite_beta;    /* compute_beta.py:26 (11) */
    int32_t max_episodes;       /* workspace capacity: largest n_ep of one mpcmmd_solve call */
    float sigma_acc, sigma_steer;     /* cem.py:167-168 */
    float ksig_steer;                 /* K_steer*sigma_steer, cem_helper.py:24,436 */
    float acc_const_noise, steer_const_noise;
    float beta_a, beta_b;             /* cem.py:24 */
    float v_min, v_max, a_max;        /* cem.py:29-31 */
    float y_lb, y_ub;                 /* cem.py:155 */
    float a_obs_sq, b_obs_sq;         /* cem.py:25 squared */
    float wheel_base, dt, steer_max, steer_rate_pen;   /* cem.py:26,40,33; cem_helper.py:249 */
    float alpha_quant, ker_wt;        /* cem.py:158,165 */
    float lamda_inv;                  /* 1/lamda, cem.py:121 */
    float alpha_mean, alpha_cov;      /* cem.py:118-119 */
    float one_minus_alpha_mean, one_minus_alpha_cov;   /* (1-alpha) evaluated in double by the host, cem_helper.py:288,291 */
    float sigma_clip;                 /* compute_beta.py:29 */
    float sigma_random;               /* cem.py:356 */
    const float *P, *Pdot, *Pddot;    /* (100,11) row-major */
    const float *Gx, *Gy;             /* x_guess affine maps (11,7), (11,8) */
    const float *Kx, *Ky;             /* projection KKT inverse rows (11,14), (11,15) */
    const float *Wfit;                /* (11,num_prime) ridge-fit matrix */
} mpcmmd_config;

/* Result of n_ep solves (device or host arrays, see the two solve entry points). */
typedef struct {
    float *cx;          /* (n_ep,11)  cx_best                       cem.py:324 */
    float *cy;          /* (n_ep,11)  cy_best                       cem.py:325 */
    float *cost_lane;   /* (n_ep,)    mmd_lane / cvar_lane / ...    cem.py:327 */
    float *cost_obs;    /* (n_ep,)    mmd_obs  / cvar_obs  / ...    cem.py:328 */
    float *beta;        /* (n_ep,num_reduced)   mmd_opt only        cem.py:329 */
    float *sigma;       /* (n_ep,)              mmd_opt only        cem.py:330 */
    float *res_beta;    /* (n_ep,maxiter_beta_cem) mmd_opt only     cem.py:331 */
} mpcmmd_out;

typedef struct mpcmmd_handle_s *mpcmmd_handle;

const char *mpcmmd_last_error(void);
int mpcmmd_version(void);

/* Environment read here: MPCMMD_PROJ = tc | tc-always selects the tensor-core projection kernel (k_project_tc: tcgen05 kind::tf32 products,
 * 1e-4 stage parity) for throughput-sized / all launches; unset = the bit-exact FP32 kernel.  See INTEGRATION.md. */
int mpcmmd_create(const mpcmmd_config *cfg, int device, mpcmmd_handle *out);
/* mpcmmd_create with the MMD kernel chosen (MPCMMD_KERNEL_*; mpcmmd_create = MPCMMD_KERNEL_LAPLACE).  The kernel is fixed for the handle's
 * lifetime: every solve and stage entry point of the handle uses it.  Unknown kinds are refused.  Both create functions refuse an
 * MPCMMD_INNER_CEM value other than auto | cta | lat | lat512 | generic (see INTEGRATION.md). */
int mpcmmd_create_with_kernel(const mpcmmd_config *cfg, int mmd_kernel, int device, mpcmmd_handle *out);
int mpcmmd_destroy(mpcmmd_handle h);

/* n_ep solves, all pointers DEVICE pointers; asynchronous on `stream` (a cudaStream_t, 0 = default).
 * idx_mpc (n_ep,) int32; init_state (n_ep,6); mean (n_ep,8); cov (n_ep,64); x_obs,y_obs (n_ep,num_obs,100); v_des (n_ep,). */
int mpcmmd_solve(mpcmmd_handle h, int cost_kind, int n_ep, const int32_t *idx_mpc, const float *init_state,
                 const float *mean, const float *cov, const float *x_obs, const float *y_obs, const float *v_des,
                 const mpcmmd_out *out, void *stream);

/* Same with HOST pointers: copies inputs up, solves, copies results back and synchronises. */
int mpcmmd_solve_host(mpcmmd_handle h, int cost_kind, int n_ep, const int32_t *idx_mpc, const float *init_state,
                      const float *mean, const float *cov, const float *x_obs, const float *y_obs, const float *v_des,
                      const mpcmmd_out *out);

/* Number of kernel launches the last mpcmmd_solve on this handle issued (graph nodes). */
int mpcmmd_last_launch_count(mpcmmd_handle h);
/* Reporting aid: name of the reduced-set inner-CEM kernel path this handle's mmd_opt launches take (static string). */
const char *mpcmmd_inner_cem_path(mpcmmd_handle h);

/* Measurement aid: re-runs the solve staged by the previous mpcmmd_solve* call launch by launch (no graph) with a
 * CUDA event after every kernel on the launching stream.  ms[5] = device milliseconds of {setup, projection,
 * rollout/risk, select, total}; n_launch[4] = launches per class.  Synchronous. */
int mpcmmd_profile_solve(mpcmmd_handle h, int cost_kind, int n_ep, float *ms, int *n_launch);

/* Monte-Carlo validation of planned trajectories: the rollout + counting part of `compute_stats`
 * (synthetic_static_obs/validation.py:134-171, synthetic_dynamic_obs/validation.py:129-165).  The reference draws its noise from
 * NumPy's legacy MT19937 stream (validation.py:43-84); those draws stay on the host, this entry point takes the PERTURBED controls.
 * All pointers are HOST pointers, float64 like the reference's NumPy arrays:
 *   acc, steer (n_ep, n_roll, num_prime); state0 (n_ep,5) = [x, y, vx, vy, psi]; x_obs_traj, y_obs_traj (n_ep, num_obs, num_prime);
 *   count, count_lane (n_ep,) int32 = max intersections over (obstacle, timestep), lane lb + ub (validation.py:156-169);
 *   x_roll, y_roll (n_ep, n_roll, num_prime) optional (both NULL to skip).
 * obs_cost_f32 = 1 evaluates the obstacle cost in float32 (static variant: x_obs_traj is a float32 jax array there), 0 in float64
 * (dynamic variant).  Synchronous. */
int mpcmmd_validate_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, double dt, double wheel_base,
                         double a_obs, double b_obs, double y_lb, double y_ub, const double *acc, const double *steer,
                         const double *state0, const double *x_obs_traj, const double *y_obs_traj, int32_t *count,
                         int32_t *count_lane, double *x_roll, double *y_roll);

/* The same validation with the noise drawn ON THE DEVICE (k_validate_noise): trajectory i's controls are perturbed with the draws of
 * np.random.seed(seed[i]) in the order of validation.py:43-84, restated in csrc/dnprng.cuh (DESIGN.md section 3 item 6).  Stream
 * consumption is NumPy's exactly; values differ from NumPy's only where CUDA's double pow / log / exp round differently from glibc's.
 * noise_kind 0 gaussian, 1 beta.  acc_plan, steer_plan (n_ep, num_prime) are the planned controls; the other inputs and the counts as
 * mpcmmd_validate_host.  Beta noise checks every shape parameter as np.random.beta does and fails with "a <= 0" / "b <= 0" before
 * anything runs.  Optional outputs (NULL to skip): acc_out, steer_out (n_ep, n_roll, num_prime) the perturbed controls (both or
 * neither); state_out (n_ep, 628) each stream after its last draw: key[624], pos, has_gauss, cached gauss as float64 bits (low word
 * first) = np.random.get_state()[1:].  All pointers are HOST pointers.  Synchronous. */
int mpcmmd_validate_seeded_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, int noise_kind,
                                double noise_level, double k_steer, double beta_a, double beta_b, double acc_const_noise,
                                double steer_const_noise, double dt, double wheel_base, double a_obs, double b_obs, double y_lb,
                                double y_ub, const uint32_t *seed, const double *acc_plan, const double *steer_plan,
                                const double *state0, const double *x_obs_traj, const double *y_obs_traj, int32_t *count,
                                int32_t *count_lane, double *acc_out, double *steer_out, uint32_t *state_out);

/* The same validation with COUNTER-BASED noise drawn by each rollout itself (k_validate_jax, DESIGN.md section 3 item 7): trajectory i's
 * noise is the JAX 0.3.23 protocol's random.beta / random.normal of (k_acc, k_steer, k_z) = split(PRNGKey(seed[i]), 3) over an
 * (n_roll, num_prime) array (csrc/drng.cuh), so a rollout's draws depend on n_roll.  Not NumPy's stream: the counts are a Monte-Carlo
 * estimate of the same quantity, not the reference's numbers.  The arguments as mpcmmd_validate_seeded_host; no shape parameter check
 * (a Beta shape of 0 gives what the sampler gives: NaN where both shapes are 0).  Fails on n_roll < 1 and n_roll * num_prime >= 2^31
 * (JAX's uint32 element counters).  Optional outputs (NULL to skip): acc_out, steer_out (n_ep, n_roll, num_prime) the perturbed
 * controls (both or neither).  All pointers are HOST pointers.  Synchronous. */
int mpcmmd_validate_threefry_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, int noise_kind,
                                  double noise_level, double k_steer, double beta_a, double beta_b, double acc_const_noise,
                                  double steer_const_noise, double dt, double wheel_base, double a_obs, double b_obs, double y_lb,
                                  double y_ub, const uint32_t *seed, const double *acc_plan, const double *steer_plan,
                                  const double *state0, const double *x_obs_traj, const double *y_obs_traj, int32_t *count,
                                  int32_t *count_lane, double *acc_out, double *steer_out);

/* Monte-Carlo RISK of each plan (DESIGN.md section 3 item 9) from the per-rollout costs
 *   c_obs  = max over (obstacle, t < num_prime) of max(0, obstacle cost)  (float32 cost in the static variant, widened; NaN propagates)
 *   c_lane = max_t max(0, y_lb - y) + max_t max(0, y - y_ub)
 * p_coll / p_lane = the fraction of rollouts with cost > 0 or NaN (NaN counts as a hit, as in the counts; the solver's saa_cost does not
 * count NaN); mean_obs; var_obs = v[lo] lw + v[hi] hw at q = alpha (n - 1) over the sorted c_obs (cvar_cost's formula in float64, no FMA);
 * cvar_obs = the mean of the c_obs >= var_obs; mmd_obs = ker_wt (S / n^2 - 2 E / n), S = sum_ij exp(-|c_i - c_j| / sigma),
 * E = sum_i exp(-c_i / sigma) (Laplace kernel; the constant term is omitted as in the solver).  Any NaN c_obs makes the four moments NaN.
 * All HOST pointers; outputs (n_ep,) unless noted.  Bit-reproducible from run to run and at any chunking. */
typedef struct {
    double alpha;                 /* VaR / CVaR level, 0..1 (the solver's alpha_quant is 0.98) */
    double ker_wt;                /* MMD scale (cem.py:165: 1000) */
    const double *sigma;          /* (n_ep,) Laplace bandwidth per plan (> 0, finite), or NULL: no MMD */
    double *p_coll, *p_lane, *mean_obs, *var_obs, *cvar_obs;   /* (n_ep,) */
    double *mmd_obs;              /* (n_ep,), required iff sigma != NULL */
    double *c_obs, *c_lane;       /* (n_ep, n_roll) per-rollout costs, optional: both or neither */
} mpcmmd_risk_out;
/* mpcmmd_validate_host's rollouts and counts (same counts) with the risk statistics; no rollout positions. */
int mpcmmd_validate_risk_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, double dt, double wheel_base,
                              double a_obs, double b_obs, double y_lb, double y_ub, const double *acc, const double *steer,
                              const double *state0, const double *x_obs_traj, const double *y_obs_traj, int32_t *count,
                              int32_t *count_lane, const mpcmmd_risk_out *risk);
/* mpcmmd_validate_threefry_host's rollouts and counts (same counts) with the risk statistics; no perturbed controls. */
int mpcmmd_validate_threefry_risk_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, int noise_kind,
                                       double noise_level, double k_steer, double beta_a, double beta_b, double acc_const_noise,
                                       double steer_const_noise, double dt, double wheel_base, double a_obs, double b_obs, double y_lb,
                                       double y_ub, const uint32_t *seed, const double *acc_plan, const double *steer_plan,
                                       const double *state0, const double *x_obs_traj, const double *y_obs_traj, int32_t *count,
                                       int32_t *count_lane, const mpcmmd_risk_out *risk);
/* The statistics of caller-supplied costs: c_obs (n_sets, n), each value >= 0 and finite or NaN; c_lane (n_sets, n) or NULL (p_lane = 0).
 * risk->c_obs / risk->c_lane are not used. */
int mpcmmd_risk_stats_host(int device, int n_sets, int n, const double *c_obs, const double *c_lane, const mpcmmd_risk_out *risk);

/* Measured FP32 FMA throughput of the device (TFLOP/s, FMA = 2 flops): the roofline denominator of the FP32-bound kernels. */
int mpcmmd_fp32_peak(int device, float *tflops, int *sm_count);
/* Measured special-function-unit peaks (thread-level operations per second / 1e9): gops[0] = ex2.approx (MUFU.EX2), gops[1] = IEEE
 * div.rn.f32, gops[2] = IEEE sqrt.rn.f32 -- the denominators for the XU-bound kernels (SURVEY.md section 8d). */
int mpcmmd_xu_peaks(int device, float *gops);
/* Exhaustive device self-check of the two IEEE shortcuts the inner-CEM kernels use (csrc/dmath.cuh): over ALL 2^32 float bit patterns,
 * mismatches[0] = dm::sqrt_rcp's root vs sqrtf, [1] = its reciprocal vs 1.0f / sqrtf, [2] = dm::div10 vs x / 10.0f (NaN == NaN).
 * All three must be 0: the shortcuts are then the IEEE operations of the arithmetic contract (S/compute_beta.py:61-63: jnp.cov, cholesky). */
int mpcmmd_selfcheck_ieee(int device, unsigned long long *mismatches /* [3], host */);

/* ---- stage entry points (teacher-forced parity tests; all DEVICE pointers, synchronous) ---- */

/* deterministic math / RNG primitives: fn 0 exp,1 log,2 log1p,3 sin,4 cos,5 tan,6 atan,7 atan2(y,x),8 erfinv, 9 exp on x <= 0, 10/11 sincos,
 * 12 Laplace kernel entry k(d = x; sigma = y) = 2^(-(d s2)) of the reduced-set inner CEM (kernel_computation.py:31-37; DESIGN.md 3.4),
 * 13 Gaussian kernel entry k(q = x; sigma = y) = 2^(-(q g2)), q a squared distance (DESIGN.md 3.8) */
int mpcmmd_math_vec(int fn, const float *x, const float *y, float *out, int n, int device);
int mpcmmd_rng_normal(uint32_t k0, uint32_t k1, int n, float *out, int device);
int mpcmmd_rng_beta(uint32_t k0, uint32_t k1, const float *a, const float *b, int n, float *out, int device);
/* copies of the constant normal tables the handle generated at create time */
int mpcmmd_get_tables(mpcmmd_handle h, float *z_init /* (B,8) */, float *theta0 /* (S,nm+1) */, float *zb_iter /* (it,S-ne,nm+1) */);

/* x_guess + projection + controls + state-cost terms for n samples (cem_helper.py:169-230,
 * projection.py:276-323, cem_helper.py:540-551,232-262).  params (n,8); beq_x (3); beq_y (4);
 * lam_x, lam_y (n,11) and s_lane (n,198) are updated in place. */
int mpcmmd_stage_project(mpcmmd_handle h, int n, const float *params, const float *beq_x, const float *beq_y, float v_des,
                         float *lam_x, float *lam_y, float *s_lane, float *cx, float *cy, float *res_norm,
                         float *acc /* (n,100) */, float *steer /* (n,100) */, float *cost_base);

/* noisy rollouts + risk for n samples (cem_helper.py:402-538, costs.py, compute_beta.py).
 * acc, steer (n,100); state0 (5); z1,z2,z3 (nr,np) normals; keys (4) beta-noise keys;
 * x_obs,y_obs (num_obs,100).  Outputs: risk, lane (n,), beta (n,nr), sigma (n,), res_beta (n,maxiter_beta_cem). */
int mpcmmd_stage_risk(mpcmmd_handle h, int cost_kind, int n, const float *acc, const float *steer, const float *state0,
                      const float *z1, const float *z2, const float *z3, const uint32_t *keys,
                      const float *x_obs, const float *y_obs, float *risk, float *lane, float *beta, float *sigma, float *res_beta);

/* The same stage with the random draws of the beta noise model INJECTED as tensors (SURVEY.md section 7 hard part 1 / 8b `set_noise`):
 * beta_acc, beta_steer (n, nr*np) are the samples of jax.random.beta(key, 2|u|, 5|u|) at cem_helper.py:427 / :432 (:492 / :497) for every
 * sample's own controls, z3 (nr*np) the common-mode normals.  No device RNG runs, so a machine that has the reference's jax==0.3.23 can feed
 * its own draws and compare everything downstream of the sampler.  (Gaussian noise: mpcmmd_stage_risk already takes z1, z2, z3.) */
int mpcmmd_stage_risk_injected(mpcmmd_handle h, int cost_kind, int n, const float *acc, const float *steer, const float *state0,
                               const float *z3, const float *beta_acc, const float *beta_steer, const float *x_obs, const float *y_obs,
                               float *risk, float *lane, float *beta, float *sigma, float *res_beta);

/* initial CEM batch of one episode (Helper.sampling_param, cem_helper.py:122-150): mean (8), cov (64) -> params (B,8). */
int mpcmmd_stage_init(mpcmmd_handle h, const float *mean, const float *cov, float *params);

/* elite selection + mean/cov update + resampling for one episode (cem.py:233-315, cem_helper.py:264-314).
 * params (B,8) is replaced by the next batch; mean (8), cov (64) updated in place; z_cem (B-5,8); sel (1) int32. */
int mpcmmd_stage_select(mpcmmd_handle h, int cost_kind, const float *res_norm, const float *risk, const float *cost_base,
                        float *params, float *mean, float *cov, const float *z_cem, int32_t *sel);

/* noise tables of one (idx_mpc, iteration): z1,z2,z3 (nr*np), z_cem ((B-5)*8), keys (4) (cem.py:225,254,302). */
int mpcmmd_stage_noise(mpcmmd_handle h, int32_t idx_mpc, int32_t iter, float *z1, float *z2, float *z3, float *z_cem, uint32_t *keys);

#ifdef __cplusplus
}
#endif
#endif
