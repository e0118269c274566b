/*
 * tests/gauss_oracle/oracle_gauss.c -- TEST INFRASTRUCTURE ONLY: the CPU oracle with the MMD kernel form as a parameter.
 *
 * The frozen oracle (oracle/oracle_mpc.c) restates the reference, whose MMD kernel is Laplace.  The opt-in Gaussian kernel
 * (DESIGN.md section 3 item 8) needs its own float32 restatement, and this file is it: it compiles the frozen oracle into the
 * same translation unit (so every helper -- rollouts, projection, selection, RNG, the KKT solve -- is the oracle's own code) and
 * restates only the three pieces the kernel form touches, with the form `ker` as an argument:
 *   gk_inner_cem  = oracle_inner_cem  with the distance table and the per-bandwidth scale of the form,
 *   gk_mmd_cost   = mmd_cost          with the scalar-cost entry of the form,
 *   gk_risk / gk_solve = oracle_risk / oracle_solve calling the two above.
 * With ker = GK_LAPLACE every function is operation for operation the frozen oracle's, and tests/test_mmd_gaussian_kernel.py
 * checks that bit for bit, which pins this copy to the oracle.  csrc/dmath.cuh dm::kern_* is the device side of the same form.
 *
 * Compile with -ffp-contract=off, like the oracle.
 */
#include "../../oracle/oracle_mpc.c"

enum { GK_LAPLACE = 0, GK_GAUSSIAN = 1 };

/* inner-CEM distance of two 22-feature rows: Laplace ascending d + |df|, Gaussian ascending fmaf(df, df, q) */
static float gk_dist(int ker, const float *Fa, const float *Fb) {
    float d = 0.0f;
    for (int f = 0; f < 2 * NV; f++) {
        if (ker == GK_GAUSSIAN) { float df = Fa[f] - Fb[f]; d = fmaf(df, df, d); }
        else d = d + fabsf(Fa[f] - Fb[f]);
    }
    return d;
}
/* per-bandwidth scale: Laplace s2 = RN(RN(1/sigma) log2 e) (om_lap_scale), Gaussian g2 = RN(RN(rinv * rinv) * RN(log2 e) / 2); entry om_lap(distance, scale) */
static om_lapscale_t gk_scale(int ker, float sigma) {
    if (ker != GK_GAUSSIAN) return om_lap_scale(sigma);
    float rinv = 1.0f / sigma;
    om_lapscale_t L;
    L.ns2 = -(rinv * rinv) * 0.72134752044448170f;      /* RN(log2(e) / 2) = RN(log2 e) / 2 exactly */
    L.dcap = 125.0f / -L.ns2;
    return L;
}
/* kernel_computation.py:67-87 compute_mmd with the scalar-cost entry om_exp(-(|dc| or dc * dc) / v), v = sigma or 2 sigma^2 */
static float gk_cost_entry(int ker, float dc, float v) { return om_exp((ker == GK_GAUSSIAN ? -(dc * dc) : -fabsf(dc)) / v); }
static float gk_mmd_cost(const ocfg_t *c, int ker, const float *beta, const float *cost, float sigma) {
    int nr = c->nr;
    float v = ker == GK_GAUSSIAN ? 2.0f * (sigma * sigma) : sigma;
    float s1 = 0.0f, s2 = 0.0f;
    for (int i = 0; i < nr; i++) {
        float t = 0.0f;
        for (int j = 0; j < nr; j++) t = fmaf(gk_cost_entry(ker, cost[i] - cost[j], v), beta[j], t);
        s1 = fmaf(beta[i], t, s1);
        float e = gk_cost_entry(ker, cost[i] - 0.0f, v), u = 0.0f;
        for (int j = 0; j < nr; j++) u = fmaf(e, c->beta_del, u);
        s2 = fmaf(beta[i], u, s2);
    }
    return c->ker_wt * (s1 - 2.0f * s2);
}

/* oracle_inner_cem with the kernel form */
static void gk_inner_cem(const ocfg_t *c, int ker, const float *F /* (nm,22) */, oinner_out_t *o) {
    int nm = c->nm, nr = c->nr, S = c->S_in, d = nm + 1, ne = c->n_el_in;
    float *th = (float *)malloc(sizeof(float) * S * d), *thn = (float *)malloc(sizeof(float) * S * d);
    float *D = (float *)malloc(sizeof(float) * nm * nm);
    float *cost = (float *)malloc(sizeof(float) * S), *betas = (float *)malloc(sizeof(float) * S * nr);
    int *idxs = (int *)malloc(sizeof(int) * S * nr), *perm = (int *)malloc(sizeof(int) * S);
    float *C = (float *)malloc(sizeof(float) * d * d), *rd = (float *)malloc(sizeof(float) * d);
    float *mean = (float *)malloc(sizeof(float) * d), *xc = (float *)malloc(sizeof(float) * ne * d);
    float *Kmix = (float *)malloc(sizeof(float) * nr * nm), *Kred = (float *)malloc(sizeof(float) * nr * nr);
    memcpy(th, c->theta0, sizeof(float) * S * d);
    if (!c->naive)
        for (int a = 0; a < nm; a++) for (int b = 0; b < nm; b++) D[a * nm + b] = gk_dist(ker, F + a * 2 * NV, F + b * 2 * NV);
    for (int it = 0; it < c->iters_in; it++) {
        for (int s = 0; s < S; s++) {
            const float *row = th + s * d;
            int *idx = idxs + s * nr;
            float sigma = row[nm], rowsum[64];
            top_abs(row, nm, nr, idx);
            om_lapscale_t ls = gk_scale(ker, sigma);
            for (int i = 0; i < nr; i++) {
                float rs = 0.0f;
                for (int m = 0; m < nm; m++) {
                    float dist = c->naive ? gk_dist(ker, F + idx[i] * 2 * NV, F + m * 2 * NV) : D[idx[i] * nm + m];
                    float k = om_lap(dist, ls);
                    Kmix[i * nm + m] = k;
                    rs = rs + k;
                }
                rowsum[i] = rs;
            }
            for (int i = 0; i < nr; i++)
                for (int j = 0; j < nr; j++) {
                    if (c->naive) { float dist = gk_dist(ker, F + idx[i] * 2 * NV, F + idx[j] * 2 * NV); Kred[i * nr + j] = om_lap(dist, ls); }
                    else Kred[i * nr + j] = Kmix[i * nm + idx[j]];
                }
            cost[s] = beta_qp(c, Kred, rowsum, betas + s * nr);
        }
        argsort_stable(cost, S, perm);
        int imin = perm[0];
        for (int e = 0; e < ne; e++) memcpy(thn + e * d, th + perm[e] * d, sizeof(float) * d);
        for (int i = 0; i < d; i++) {
            float s = 0.0f;
            for (int e = 0; e < ne; e++) s = s + thn[e * d + i];
            mean[i] = s / (float)ne;
        }
        for (int e = 0; e < ne; e++) for (int i = 0; i < d; i++) xc[e * d + i] = thn[e * d + i] - mean[i];
        for (int i = 0; i < d; i++)
            for (int j = 0; j <= i; j++) {
                float a = 0.0f;
                for (int e = 0; e < ne; e++) a = fmaf(xc[e * d + i], xc[e * d + j], a);
                a = a / (float)(ne - 1);
                if (i == j) a = a + 0.05f;
                C[i * d + j] = a;
            }
        chol_inplace(C, d, d, rd);
        const float *z = c->zb_iter + (size_t)it * (S - ne) * d;
        for (int r = 0; r < S - ne; r++)
            for (int i = 0; i < d; i++) thn[(ne + r) * d + i] = mvn_elem(C, d, i, z + r * d, mean[i]);
        for (int s = 0; s < S; s++) { float v = thn[s * d + nm]; thn[s * d + nm] = (v != v) ? v : (v > c->sigma_clip ? v : c->sigma_clip); }
        o->res[it] = cost[imin];
        if (it == c->iters_in - 1) {
            for (int i = 0; i < nr; i++) { o->beta[i] = betas[imin * nr + i]; o->idx[i] = idxs[imin * nr + i]; }
            o->sigma = thn[imin * d + nm];
        }
        float *tmp = th; th = thn; thn = tmp;
    }
    free(th); free(thn); free(D); free(cost); free(betas); free(idxs); free(perm); free(C); free(rd); free(mean); free(xc); free(Kmix); free(Kred);
}

/* oracle_risk with the kernel form (its cvar / saa branches do not depend on it) */
void gk_risk(const ocfg_t *c, int ker, int cost_kind, const float *acc, const float *steer, const float *st0,
             const onoise_t *nz, const float *x_obs, const float *y_obs, orisk_out_t *o) {
    int nr = c->nr, np = c->np, nm = c->nm;
    int R = (cost_kind == COST_MMD_OPT) ? nm : nr;
    float *an = (float *)malloc(sizeof(float) * nr * np), *sn = (float *)malloc(sizeof(float) * nr * np);
    float *xr = (float *)malloc(sizeof(float) * R * np), *yr = (float *)malloc(sizeof(float) * R * np);
    noisy_controls(c, acc, steer, nz, an, sn);
    for (int m = 0; m < R; m++) {
        int ia = (cost_kind == COST_MMD_OPT) ? m / nr : m, is = (cost_kind == COST_MMD_OPT) ? m % nr : m;
        rollout_one(c, an + ia * np, sn + is * np, st0, xr + m * np, yr + m * np);
    }
    float cst[64], lb[64], ub[64];
    memset(o, 0, sizeof *o);
    if (cost_kind == COST_MMD_OPT) {
        float *F = (float *)malloc(sizeof(float) * nm * 2 * NV);
        for (int m = 0; m < nm; m++)
            for (int k = 0; k < NV; k++) {
                float ax = 0.0f, ay = 0.0f;
                for (int t = 0; t < np; t++) { ax = fmaf(c->Wfit[k * np + t], xr[m * np + t], ax); ay = fmaf(c->Wfit[k * np + t], yr[m * np + t], ay); }
                F[m * 2 * NV + k] = ax; F[m * 2 * NV + NV + k] = ay;
            }
        oinner_out_t in;
        gk_inner_cem(c, ker, F, &in);
        free(F);
        for (int i = 0; i < nr; i++) {
            int m = in.idx[i];
            o->red_idx[i] = m; o->beta[i] = in.beta[i];
            cst[i] = fbar_max(c, xr + m * np, yr + m * np, x_obs, y_obs);
            lane_max(c, yr + m * np, &lb[i], &ub[i]);
        }
        o->sigma = in.sigma;
        for (int i = 0; i < c->iters_in; i++) o->res_beta[i] = in.res[i];
        o->risk = gk_mmd_cost(c, ker, o->beta, cst, o->sigma);
        o->lane = gk_mmd_cost(c, ker, o->beta, lb, o->sigma) + gk_mmd_cost(c, ker, o->beta, ub, o->sigma);
    } else {
        for (int i = 0; i < nr; i++) {
            o->red_idx[i] = i;
            cst[i] = fbar_max(c, xr + i * np, yr + i * np, x_obs, y_obs);
            lane_max(c, yr + i * np, &lb[i], &ub[i]);
        }
        if (cost_kind == COST_MMD_RANDOM) {
            for (int i = 0; i < nr; i++) o->beta[i] = c->beta_del;
            o->sigma = c->sigma_random;
            o->risk = gk_mmd_cost(c, ker, o->beta, cst, o->sigma);
            o->lane = 0.0f;
        } else if (cost_kind == COST_CVAR) {
            o->risk = cvar_cost(c, cst);
            o->lane = cvar_cost(c, lb) + cvar_cost(c, ub);
        } else {
            o->risk = saa_cost(c, cst);
            float sl = 0.0f, su = 0.0f;
            for (int i = 0; i < nr; i++) { sl = sl + (lb[i] > 0.0f ? 1.0f : 0.0f); su = su + (ub[i] > 0.0f ? 1.0f : 0.0f); }
            o->lane = (sl + su) / (float)nr;
        }
    }
    for (int i = 0; i < nr; i++) o->red_cost[i] = cst[i];
    free(an); free(sn); free(xr); free(yr);
}

/* oracle_solve with the kernel form */
typedef struct { osample_job_t j; int ker; } gk_job_t;
static void *gk_worker(void *arg) {
    gk_job_t *g = (gk_job_t *)arg;
    osample_job_t *j = &g->j;
    for (int b = j->b0; b < j->b1; b++) {
        oracle_project(j->c, j->params + b * NP_, j->beq_x, j->beq_y, j->v_des, j->lam_x + b * NV, j->lam_y + b * NV, j->s_lane + b * 2 * NL, &j->pr[b]);
        gk_risk(j->c, g->ker, j->cost_kind, j->pr[b].acc, j->pr[b].steer, j->st0, j->nz, j->x_obs, j->y_obs, &j->rk[b]);
    }
    return NULL;
}
int gk_solve(const ocfg_t *c, int ker, int cost_kind, int32_t idx_mpc, const float *init_state, const float *mean0,
             const float *cov0, const float *x_obs, const float *y_obs, float v_des, osolve_out_t *out) {
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
    orisk_out_t *rk = (orisk_out_t *)malloc(sizeof(orisk_out_t) * B);
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
            pthread_t th[256]; gk_job_t jobs[256];
            for (int k = 0; k < nt; k++) {
                osample_job_t j = {c, cost_kind, params, beq_x, beq_y, v_des, lam_x, lam_y, s_lane, pr, rk, st0, &nz, x_obs, y_obs,
                                   (int)((long)B * k / nt), (int)((long)B * (k + 1) / nt)};
                jobs[k].j = j; jobs[k].ker = ker;
                if (nt > 1) pthread_create(&th[k], NULL, gk_worker, &jobs[k]); else gk_worker(&jobs[k]);
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
            out->cost_lane = rk[s].lane; out->cost_obs = rk[s].risk;
            for (int i = 0; i < nr; i++) out->beta[i] = rk[s].beta[i];
            out->sigma = rk[s].sigma;
            for (int i = 0; i < c->iters_in; i++) out->res_beta[i] = rk[s].res_beta[i];
            out->sel_last = s;
        }
        float *tmp = params; params = params_next; params_next = tmp;
    }
    free(params); free(params_next); free(lam_x); free(lam_y); free(s_lane); free(pr); free(rk);
    free(res_norm); free(risk); free(base); free(z1); free(z2); free(z3); free(z_cem);
    return 0;
}

/* the inner-CEM entry k(q = x[i]; sigma = y[i]) of the form */
void gk_entry_vec(int ker, const float *x, const float *y, float *out, int n) {
    for (int i = 0; i < n; i++) out[i] = om_lap(x[i], gk_scale(ker, y[i]));
}
