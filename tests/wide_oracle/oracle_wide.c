/*
 * tests/wide_oracle/oracle_wide.c -- TEST INFRASTRUCTURE ONLY: the CPU oracle for cvar / saa / mmd_random at any num_reduced.
 *
 * The frozen oracle (oracle/oracle_mpc.c) keeps per-sample results in fixed [64] arrays (cvar_cost's permutation, oracle_risk's cost
 * arrays, orisk_out_t, osolve_out_t), so it stops at num_reduced 64.  The formulas themselves are generic in num_reduced (DESIGN.md section
 * 3), and this file restates, with heap arrays, only the pieces that hold those arrays:
 *   wd_cvar  = cvar_cost                        (the same stable NaN-last argsort, quantile and sequential tail sum),
 *   wd_risk  = oracle_risk / gk_risk without the mmd_opt branch, with the MMD kernel form as an argument,
 *   wd_solve = oracle_solve / gk_solve calling wd_risk.
 * It includes tests/gauss_oracle/oracle_gauss.c, which compiles the frozen oracle into the same translation unit, so every other helper
 * (noise tables, Beta sampler, rollouts, obstacle and lane maxima, projection, selection, gk_mmd_cost) is the oracle's own code.  For
 * num_reduced <= 64 tests/test_wide_oracle.py checks wd_risk and wd_solve against the frozen oracle bit for bit, which pins this copy to it.
 *
 * Compile with -ffp-contract=off, like the oracle.
 */
#include "../gauss_oracle/oracle_gauss.c"

/* cvar_cost of n values: jnp.quantile linear interpolation + the mean of the v >= var (costs.py:213-220) */
float wd_cvar(float alpha_quant, const float *v, int nr) {
    int *perm = (int *)malloc(sizeof(int) * (nr > 0 ? nr : 1));
    argsort_stable(v, nr, perm);
    float q = alpha_quant * (float)(nr - 1);
    float lo = floorf(q), hi = ceilf(q);
    float hw = q - lo, lw = 1.0f - hw;
    int ilo = (int)lo, ihi = (int)hi;
    if (ilo < 0) ilo = 0; if (ilo > nr - 1) ilo = nr - 1;
    if (ihi < 0) ihi = 0; if (ihi > nr - 1) ihi = nr - 1;
    float var = v[perm[ilo]] * lw + v[perm[ihi]] * hw;
    float s = 0.0f; int n = 0;
    for (int i = 0; i < nr; i++) if (v[i] >= var) { s = s + v[i]; n++; }
    free(perm);
    return n > 0 ? s / (float)n : 0.0f;
}
/* saa_cost of n values */
float wd_saa(const float *v, int nr) {
    float s = 0.0f;
    for (int i = 0; i < nr; i++) s = s + (v[i] > 0.0f ? 1.0f : 0.0f);
    return s / (float)nr;
}

/* one sample's risk stage; beta / red_cost (nr) are optional outputs */
typedef struct { float risk, lane, sigma; float *beta, *red_cost; } wrisk_out_t;

void wd_risk(const ocfg_t *c, int ker, int cost_kind, const float *acc, const float *steer, const float *st0,
             const onoise_t *nz, const float *x_obs, const float *y_obs, wrisk_out_t *o) {
    int nr = c->nr, np = c->np;
    float *an = (float *)malloc(sizeof(float) * nr * np), *sn = (float *)malloc(sizeof(float) * nr * np);
    float *xr = (float *)malloc(sizeof(float) * nr * np), *yr = (float *)malloc(sizeof(float) * nr * np);
    float *cst = (float *)malloc(sizeof(float) * nr), *lb = (float *)malloc(sizeof(float) * nr), *ub = (float *)malloc(sizeof(float) * nr);
    float *beta = (float *)malloc(sizeof(float) * nr);
    noisy_controls(c, acc, steer, nz, an, sn);
    for (int m = 0; m < nr; m++) rollout_one(c, an + m * np, sn + m * np, st0, xr + m * np, yr + m * np);
    for (int i = 0; i < nr; i++) {
        cst[i] = fbar_max(c, xr + i * np, yr + i * np, x_obs, y_obs);
        lane_max(c, yr + i * np, &lb[i], &ub[i]);
        beta[i] = 0.0f;
    }
    o->sigma = 0.0f;
    if (cost_kind == COST_MMD_RANDOM) {          /* cem.py:355-356, 404-424: beta = 1/nr, sigma = 0.01, lane = 0 */
        for (int i = 0; i < nr; i++) beta[i] = c->beta_del;
        o->sigma = c->sigma_random;
        o->risk = gk_mmd_cost(c, ker, beta, cst, o->sigma);
        o->lane = 0.0f;
    } else if (cost_kind == COST_CVAR) {         /* costs.py:206-221, 137-158 */
        o->risk = wd_cvar(c->alpha_quant, cst, nr);
        o->lane = wd_cvar(c->alpha_quant, lb, nr) + wd_cvar(c->alpha_quant, ub, nr);
    } else {                                     /* costs.py:223-234, 160-171 */
        o->risk = wd_saa(cst, nr);
        float sl = 0.0f, su = 0.0f;
        for (int i = 0; i < nr; i++) { sl = sl + (lb[i] > 0.0f ? 1.0f : 0.0f); su = su + (ub[i] > 0.0f ? 1.0f : 0.0f); }
        o->lane = (sl + su) / (float)nr;
    }
    if (o->beta) memcpy(o->beta, beta, sizeof(float) * nr);
    if (o->red_cost) memcpy(o->red_cost, cst, sizeof(float) * nr);
    free(an); free(sn); free(xr); free(yr); free(cst); free(lb); free(ub); free(beta);
}

/* the solve: oracle_solve's loop with wd_risk; beta (nr) optional */
typedef struct { float cx[NV], cy[NV], cost_lane, cost_obs, sigma; int32_t sel_last; } wsolve_out_t;
typedef struct { const ocfg_t *c; int ker, cost_kind; const float *params, *beq_x, *beq_y; float v_des; float *lam_x, *lam_y, *s_lane;
                 oproj_out_t *pr; wrisk_out_t *rk; const float *st0; const onoise_t *nz; const float *x_obs, *y_obs; int b0, b1; } wd_job_t;
static void *wd_worker(void *arg) {
    wd_job_t *j = (wd_job_t *)arg;
    for (int b = j->b0; b < j->b1; b++) {
        oracle_project(j->c, j->params + b * NP_, j->beq_x, j->beq_y, j->v_des, j->lam_x + b * NV, j->lam_y + b * NV, j->s_lane + b * 2 * NL, &j->pr[b]);
        wd_risk(j->c, j->ker, j->cost_kind, j->pr[b].acc, j->pr[b].steer, j->st0, j->nz, j->x_obs, j->y_obs, &j->rk[b]);
    }
    return NULL;
}
int wd_solve(const ocfg_t *c, int ker, int cost_kind, int32_t idx_mpc, const float *init_state, const float *mean0,
             const float *cov0, const float *x_obs, const float *y_obs, float v_des, wsolve_out_t *out, float *beta_out) {
    int B = c->B, np = c->np, nr = c->nr;
    float beq_x[3] = {init_state[0], init_state[2], init_state[4]};
    float beq_y[4] = {init_state[1], init_state[3], init_state[5], 0.0f};
    float st0[5] = {init_state[0], init_state[1], init_state[2], init_state[3], om_atan2(init_state[3], init_state[2])};
    float mean[NP_], cov[NP_ * NP_];
    memcpy(mean, mean0, sizeof mean); memcpy(cov, cov0, sizeof cov);
    float *params = (float *)malloc(sizeof(float) * B * NP_), *params_next = (float *)malloc(sizeof(float) * B * NP_);
    float *lam_x = (float *)calloc((size_t)B * NV, sizeof(float)), *lam_y = (float *)calloc((size_t)B * NV, sizeof(float));
    float *s_lane = (float *)calloc((size_t)B * 2 * NL, sizeof(float));
    oproj_out_t *pr = (oproj_out_t *)malloc(sizeof(oproj_out_t) * B);
    wrisk_out_t *rk = (wrisk_out_t *)calloc((size_t)B, sizeof(wrisk_out_t));
    float *betas = (float *)malloc(sizeof(float) * (size_t)B * nr);
    for (int b = 0; b < B; b++) rk[b].beta = betas + (size_t)b * nr;
    float *res_norm = (float *)malloc(sizeof(float) * B), *risk = (float *)malloc(sizeof(float) * B), *base = (float *)malloc(sizeof(float) * B);
    int n = nr * np;
    float *z1 = (float *)malloc(sizeof(float) * n), *z2 = (float *)malloc(sizeof(float) * n), *z3 = (float *)malloc(sizeof(float) * n);
    float *z_cem = (float *)malloc(sizeof(float) * (B - c->n_el) * NP_);
    oracle_sample_params(c, mean, cov, c->z_init, B, params);
    for (int it = 0; it < c->iters; it++) {
        uint32_t keys[4];
        oracle_noise_tables(c, idx_mpc, it, z1, z2, z3, z_cem, keys);
        onoise_t nz = {z1, z2, z3, {keys[0], keys[1]}, {keys[2], keys[3]}, NULL, NULL};
        {
            int nt = g_oracle_threads < 1 ? 1 : (g_oracle_threads > 256 ? 256 : g_oracle_threads);
            if (nt > B) nt = B;
            pthread_t th[256]; wd_job_t jobs[256];
            for (int k = 0; k < nt; k++) {
                wd_job_t j = {c, ker, cost_kind, params, beq_x, beq_y, v_des, lam_x, lam_y, s_lane, pr, rk, st0, &nz, x_obs, y_obs,
                              (int)((long)B * k / nt), (int)((long)B * (k + 1) / nt)};
                jobs[k] = j;
                if (nt > 1) pthread_create(&th[k], NULL, wd_worker, &jobs[k]); else wd_worker(&jobs[k]);
            }
            if (nt > 1) for (int k = 0; k < nt; k++) pthread_join(th[k], NULL);
            for (int b = 0; b < B; b++) { res_norm[b] = pr[b].res_norm; risk[b] = rk[b].risk; base[b] = pr[b].cost_base; }
        }
        oselect_out_t so;
        oracle_select(c, res_norm, risk, base, params, params_next, mean, cov, z_cem, &so);
        if (it == c->iters - 1) {
            int s = so.sel;
            memset(out, 0, sizeof *out);
            memcpy(out->cx, pr[s].cx, sizeof out->cx); memcpy(out->cy, pr[s].cy, sizeof out->cy);
            out->cost_lane = rk[s].lane; out->cost_obs = rk[s].risk; out->sigma = rk[s].sigma;
            if (beta_out) memcpy(beta_out, rk[s].beta, sizeof(float) * nr);
            out->sel_last = s;
        }
        float *tmp = params; params = params_next; params_next = tmp;
    }
    free(params); free(params_next); free(lam_x); free(lam_y); free(s_lane); free(pr); free(rk); free(betas);
    free(res_norm); free(risk); free(base); free(z1); free(z2); free(z3); free(z_cem);
    return 0;
}
