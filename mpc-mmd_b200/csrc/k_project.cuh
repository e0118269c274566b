// k_project.cuh -- noise tables, batch initialisation and the per-sample projection kernel.
//
// k_project replaces, per CEM sample (one warp each):
//   Helper.compute_x_guess            reference S/optimizer/cem_helper.py:169-230
//   Projection.compute_projection     S/optimizer/projection.py:276-323 (+ :52-121, :123-185, :193-274)
//   Helper.compute_controls           S/optimizer/cem_helper.py:540-551
//   the risk-independent terms of Helper.compute_cost   S/optimizer/cem_helper.py:232-262
// Lane l of the warp owns the knots t = l, l+32, l+64, l+96; "transposed" products (P^T r) are
// formed by lanes 0..21 (11 x-coefficients, 11 y-coefficients) as ascending-t fma chains, which
// is the summation order the arithmetic contract fixes.
#pragma once
#include "common.cuh"

// ---------------------------------------------------------------------------------------------
// noise tables for every (episode, outer iteration): cem.py:225,254,302; cem_helper.py:405-443
__global__ void k_noise(DCfg c, DWork w, int n_ep, int it0, int n_it) {
    const int blk = blockIdx.x;               // e * n_it + (it - it0)
    const int e = blk / n_it, it = it0 + blk % n_it;
    if (e >= n_ep) return;
    const int n = c.nr * c.np, ncem = (c.B - c.n_el) * NPAR;
    dr::Key key; key.k0 = 0u; key.k1 = (uint32_t)(3 * w.idx_mpc[e] + 5 * it + 7);
    const dr::Key k1 = dr::split0(key), k2 = dr::split0(k1), k3 = dr::split0(k2);
    const size_t slot = (size_t)e * c.iters + it;
    float* z1 = w.z1 + slot * n; float* z2 = w.z2 + slot * n; float* z3 = w.z3 + slot * n;
    float* zc = w.zcem + slot * ncem;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        if (c.noise_kind == 0) {
            z1[i] = dr::normal_elem(k1, (uint32_t)n, (uint32_t)i);
            z2[i] = dr::normal_elem(k2, (uint32_t)n, (uint32_t)i);
        }
        z3[i] = dr::normal_elem(k3, (uint32_t)n, (uint32_t)i);
    }
    for (int i = threadIdx.x; i < ncem; i += blockDim.x) zc[i] = dr::normal_elem(k2, (uint32_t)ncem, (uint32_t)i);   // [Q6]
    if (c.noise_kind == 1 && w.btab) {        // candidates of the Beta rejection sampler, shared by the B samples of the episode [Q5]
        float* bt = w.btab + slot * (size_t)(4 * GT_FIELDS) * n;
        for (int i = threadIdx.x; i < 4 * n; i += blockDim.x) {
            const int stream = i / n, el = i % n;
            dr::gamma_table_fill(dr::gamma_stream_key(k1, k2, stream), (uint32_t)n, (uint32_t)el, bt + (size_t)stream * GT_FIELDS * n + el);
        }
    }
    if (threadIdx.x == 0) {
        uint32_t* k = w.keys + slot * 4;
        k[0] = k1.k0; k[1] = k1.k1; k[2] = k2.k0; k[3] = k2.k1;
    }
}

// generic table of normals: out[i] = normal(key, (n,))[i]
__global__ void k_normal_table(uint32_t k0, uint32_t k1, int n, float* out) {
    dr::Key key; key.k0 = k0; key.k1 = k1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i] = dr::normal_elem(key, (uint32_t)n, (uint32_t)i);
}
__global__ void k_beta_table(uint32_t k0, uint32_t k1, const float* a, const float* b, int n, float* out) {
    dr::Key key; key.k0 = k0; key.k1 = k1;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
        out[i] = dr::beta_elem(key, (uint32_t)n, (uint32_t)i, a[i], b[i]);
}
__global__ void k_math_vec(int fn, const float* x, const float* y, float* out, int n) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        float v;
        switch (fn) {
            case 0: v = dm::exp_(x[i]); break;
            case 1: v = dm::log_(x[i]); break;
            case 2: v = dm::log1p_(x[i]); break;
            case 3: v = dm::sin_(x[i]); break;
            case 4: v = dm::cos_(x[i]); break;
            case 5: v = dm::tan_(x[i]); break;
            case 6: v = dm::atan_(x[i]); break;
            case 7: v = dm::atan2_(y[i], x[i]); break;
            case 8: v = dr::erfinv32(x[i]); break;
            case 9: v = dm::exp_nonpos(x[i]); break;
            case 10: { float s, cc; dm::sincos_(x[i], s, cc); v = s; } break;
            case 11: { float s, cc; dm::sincos_(x[i], s, cc); v = cc; } break;
            case 12: v = dm::lap_(x[i], dm::lap_scale(y[i])); break;          // Laplace kernel entry k(d = x; sigma = y) of the reduced-set inner CEM
            case 13: v = dm::lap_(x[i], dm::kern_scale<dm::KER_GAUSSIAN>(y[i])); break;      // Gaussian kernel entry k(q = x; sigma = y), q a squared distance
            default: v = DM_NAN;
        }
        out[i] = v;
    }
}
// [iter][row][col] -> [iter][col][row]
__global__ void k_transpose_tables(const float* src, float* dst, int n_it, int rows, int cols) {
    const int n = n_it * rows * cols;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int it = i / (rows * cols), rem = i % (rows * cols), r = rem / cols, q = rem % cols;
        dst[(size_t)it * rows * cols + (size_t)q * rows + r] = src[i];
    }
}
// theta0 = sqrt(20) * z with the bandwidth column clipped (compute_beta.py:41-49, :20-24)
__global__ void k_theta0(const float* z, int S, int d, float sigma_clip, float* out) {
    const float s20 = sqrtf(20.0f);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < S * d; i += gridDim.x * blockDim.x) {
        float v = s20 * z[i];
        if (i % d == d - 1) v = (v != v) ? v : (v > sigma_clip ? v : sigma_clip);
        out[i] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// sampling of a CEM batch from N(mean, cov): multivariate_normal(cholesky) + speed clip
// (cem_helper.py:122-150 and :292-312).  One thread block; L (8x8) is built by thread 0.
__device__ __forceinline__ void sample_batch(const DCfg& c, const float* mean, const float* covL /* smem L */, const float* z,
                                             int rows, float* out) {
    for (int i = threadIdx.x; i < rows * NPAR; i += blockDim.x) {
        const int r = i / NPAR, col = i % NPAR;
        float v = mvn_elem(covL, NPAR, col, z + r * NPAR, mean[col]);
        out[i] = (col < 4) ? dm::clip_(v, c.v_min, c.v_max) : v;
    }
}

// start of a solve (cem.py:206-219): zero multipliers / slacks, copy mean/cov, draw the first batch
__global__ void k_init(DCfg c, DWork w, int n_ep) {
    const int e = blockIdx.x;
    if (e >= n_ep) return;
    __shared__ float L[NPAR * NPAR], rd[NPAR], mean[NPAR];
    const int B = c.B;
    if (threadIdx.x < NPAR * NPAR) { float v = w.cov0[e * 64 + threadIdx.x]; L[threadIdx.x] = v; w.cov[e * 64 + threadIdx.x] = v; }
    if (threadIdx.x < NPAR) { float v = w.mean0[e * NPAR + threadIdx.x]; mean[threadIdx.x] = v; w.mean[e * NPAR + threadIdx.x] = v; }
    __syncthreads();
    if (threadIdx.x == 0) chol_serial(L, NPAR, NPAR, rd);
    __syncthreads();
    sample_batch(c, mean, L, c.z_init, B, w.params + (size_t)e * B * NPAR);
    for (int i = threadIdx.x; i < B * NV; i += blockDim.x) { w.lam_x[(size_t)e * B * NV + i] = 0.0f; w.lam_y[(size_t)e * B * NV + i] = 0.0f; }
    for (int i = threadIdx.x; i < B * 2 * NL; i += blockDim.x) w.s_lane[(size_t)e * B * 2 * NL + i] = 0.0f;
}

// ---------------------------------------------------------------------------------------------
// projection

#define PROJ_WARPS 8
#define PROJ_CONST_FLOATS (3 * T_ * NV + 77 + 88 + 154 + 165)      // P,Pd,Pdd,Gx,Gy,Kx,Ky
#define PROJ_WARP_FLOATS (24 + 32 + 24 + 9 * T_ + 200)              // cb, rhs, cc, V0..V8, LA (= LB: the lane right-hand side is dead before the lane residual is written)
#define PROJ_SMEM_BYTES ((PROJ_CONST_FLOATS + PROJ_WARPS * PROJ_WARP_FLOATS) * 4)

struct ProjArgs {           // one batch of samples; sample g = e * B + b uses per-episode boundary data
    int n_samples, B;       // B: samples per episode (for indexing the per-episode arrays)
    const float* params;    // [n][8]
    const float* beq_x;     // [E][3]   (x_init, vx_init, ax_init)
    const float* beq_y;     // [E][4]
    const float* v_des;     // [E]
    float *lam_x, *lam_y;   // [n][11]
    float* s_lane;          // [n][198]
    float *cx, *cy;         // [n][11]
    float *res_norm, *cost_base;   // [n]
    float *acc, *steer;     // [n][100]
    int dbg;                // k_project_tc only: 1 / 2 = dump the pass-1 products instead of the results (tools/proj_tc_probe.py)
};

__device__ __forceinline__ float unwrap_corr(float dd) {     // jnp.unwrap phase correction for one difference
    const float PI = 3.14159265358979323846f, TWO_PI = 6.28318530717958647692f;
    if (fabsf(dd) < PI) return 0.0f;
    float a = dd + PI;
    float r = fmodf(a, TWO_PI);
    if (r != 0.0f && r < 0.0f) r += TWO_PI;
    float ddmod = r - PI;
    if (ddmod == -PI && dd > 0.0f) ddmod = PI;
    return ddmod - dd;
}
// polar re-parametrisation of one (vx,vy) pair: returns d*cos, d*sin for clip bounds [lo,hi] (projection.py:80-99 / 224-243)
__device__ __forceinline__ void polar_clip(float alpha, float wx, float wy, float lo, float hi, float& bx, float& by) {
    float s, cs; dm::sincos_(alpha, s, cs);
    float c1 = cs * cs + s * s;
    float c2 = wx * cs + wy * s;
    float d = dm::clip_(c2 / c1, lo, hi);
    bx = d * cs; by = d * s;
}

// two dot11 chains over one basis row (x coefficients c[0..10], y coefficients c[11..21] held in registers): the same ascending fma chain per
// output as dot11, half the shared-memory loads
__device__ __forceinline__ void dot11x2(const float* row, const float (&c)[2 * NV], float& ox, float& oy) {
    float ax = 0.0f, ay = 0.0f;
#pragma unroll
    for (int k = 0; k < NV; k++) { const float p = row[k]; ax = fmaf(p, c[k], ax); ay = fmaf(p, c[NV + k], ay); }
    ox = ax; oy = ay;
}

__global__ void __launch_bounds__(PROJ_WARPS * 32, 4) k_project(DCfg c, ProjArgs a) {
    extern __shared__ __align__(128) float sm[];
    static_assert(PROJ_CONST_FLOATS % 4 == 0 && PROJ_WARP_FLOATS % 4 == 0, "the per-warp vectors are read with 16-byte loads");
    float* sP = sm; float* sPd = sP + T_ * NV; float* sPdd = sPd + T_ * NV;
    float* sGx = sPdd + T_ * NV; float* sGy = sGx + 77; float* sKx = sGy + 88; float* sKy = sKx + 154;
    // the 15 KB of constant matrices arrive as ONE TMA bulk copy (cp.async.bulk + mbarrier) instead of ~15 loads and stores per thread
    __shared__ __align__(8) unsigned long long cbar;
    static_assert((PROJ_CONST_FLOATS * 4) % 16 == 0, "bulk copies move multiples of 16 bytes");
    if (threadIdx.x == 0) mbar_init(&cbar, 1);
    __syncthreads();
    if (threadIdx.x == 0) bulk_g2s(sm, c.proj_const, PROJ_CONST_FLOATS * 4, &cbar);
    mbar_wait(&cbar, 0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int g = blockIdx.x * PROJ_WARPS + warp;
    if (g >= a.n_samples) return;                      // whole warp exits together; no block sync below
    const int e = g / a.B;
    float* ws = sm + PROJ_CONST_FLOATS + warp * PROJ_WARP_FLOATS;
    float* cb = ws; float* rhs = cb + 24; float* cc = rhs + 32;
    float* V0 = cc + 24; float* V1 = V0 + T_; float* V2 = V1 + T_; float* V3 = V2 + T_; float* V4 = V3 + T_;
    float* V5 = V4 + T_; float* V6 = V5 + T_; float* V7 = V6 + T_; float* V8 = V7 + T_;
    float* LA = V8 + T_; float* LB = LA;
    const float* par = a.params + (size_t)g * NPAR;
    const float* bqx = a.beq_x + e * 3; const float* bqy = a.beq_y + e * 4;
    const bool isx = lane < NV; const int j = isx ? lane : lane - NV;      // coefficient index for lanes < 22

    // ---- x_guess: affine map of (params, boundary values)  [cem_helper.py:169-230, folded]
    if (lane < 2 * NV) {
        float acc = 0.0f;
        if (isx) {
#pragma unroll
            for (int k = 0; k < 7; k++) acc = fmaf(sGx[j * 7 + k], (k < 4) ? par[k] : bqx[k - 4], acc);
        } else {
#pragma unroll
            for (int k = 0; k < 8; k++) acc = fmaf(sGy[j * 8 + k], (k < 4) ? par[4 + k] : bqy[k - 4], acc);
        }
        cb[lane] = acc;
    }
    __syncwarp();
    // ---- guess derivatives + raw angles  [projection.py:285-289, :77, :91]
    float cr[2 * NV];                                 // the 22 coefficients in registers: every basis-row element is loaded once and feeds the x and the y chain
#pragma unroll
    for (int k = 0; k < 2 * NV; k++) cr[k] = cb[k];
    for (int t = lane; t < T_; t += 32) {
        float xdg, ydg, xddg, yddg;
        dot11x2(sPd + t * NV, cr, xdg, ydg);
        dot11x2(sPdd + t * NV, cr, xddg, yddg);
        V0[t] = xdg; V1[t] = ydg; V2[t] = xddg; V3[t] = yddg;
        V4[t] = dm::atan2_(ydg, xdg); V5[t] = dm::atan2_(yddg, xddg);
    }
    __syncwarp();
    // ---- jnp.unwrap along time
    bool anyc = false;
    for (int t = lane; t < T_; t += 32) {
        float cv = 0.0f, ca = 0.0f;
        if (t >= 1) { cv = unwrap_corr(V4[t] - V4[t - 1]); ca = unwrap_corr(V5[t] - V5[t - 1]); }
        V6[t] = cv; V7[t] = ca;
        anyc |= (cv != 0.0f) || (ca != 0.0f);
    }
    anyc = __any_sync(FULL, anyc);
    __syncwarp();
    if (anyc) {                                       // rare: sequential cumulative sum, as the contract states
        if (lane < 2) { float* Vc = lane ? V7 : V6; float cs = 0.0f; for (int t = 1; t < T_; t++) { cs = cs + Vc[t]; Vc[t] = cs; } }
        __syncwarp();
    }
    // ---- initial_alpha_d_obs: polar step, residuals  [projection.py:73-113]
    for (int t = lane; t < T_; t += 32) {
        float av = (t >= 1) ? V4[t] + V6[t] : V4[t];
        float aa = (t >= 1) ? V5[t] + V7[t] : V5[t];
        float xdg = V0[t], ydg = V1[t], xddg = V2[t], yddg = V3[t];
        float bvx, bvy, bax, bay;
        polar_clip(av, xdg, ydg, c.v_min, c.v_max, bvx, bvy);
        polar_clip(aa, xddg, yddg, 0.0f, c.a_max, bax, bay);
        V4[t] = xddg - bax; V5[t] = yddg - bay; V6[t] = xdg - bvx; V7[t] = ydg - bvy;    // r_ax, r_ay, r_vx, r_vy
        V0[t] = bax; V1[t] = bay; V2[t] = bvx; V3[t] = bvy;                                // b_*_ineq of compute_x
    }
    // lane-constraint right-hand side  b_lane_bound - s_lane  [projection.py:127-131]
    float* sl = a.s_lane + (size_t)g * 2 * NL;
    for (int i = lane; i < 2 * NL; i += 32) LA[i] = ((i < NL) ? c.b_lane_ub : c.b_lane_lb) - sl[i];
    __syncwarp();
    // ---- multiplier update + lincost + KKT solve  [projection.py:115-119, 158-171]
    float lam = 0.0f;
    if (lane < 2 * NV) {
        float* lamg = (isx ? a.lam_x : a.lam_y) + (size_t)g * NV + j;
        lam = *lamg;
        const float* rA = isx ? V4 : V5; const float* rV = isx ? V6 : V7;
        const float* bA = isx ? V0 : V1; const float* bV = isx ? V2 : V3;
        // five independent ascending chains advance together (each keeps its own order): P^T r (2), P^T b (2) and the first 99 terms of the lane chain
        float a1 = 0.0f, a2 = 0.0f, b1 = 0.0f, b2 = 0.0f, a3 = 0.0f;
        for (int t = 0; t < T_; t += 4) {             // the per-knot vectors are 16-byte aligned: one LDS.128 feeds four steps of a chain
            const float4 ra = *reinterpret_cast<const float4*>(rA + t), rv = *reinterpret_cast<const float4*>(rV + t);
            const float4 ba = *reinterpret_cast<const float4*>(bA + t), bv = *reinterpret_cast<const float4*>(bV + t);
            const float4 la = *reinterpret_cast<const float4*>(LA + t);
            const float ra_[4] = {ra.x, ra.y, ra.z, ra.w}, rv_[4] = {rv.x, rv.y, rv.z, rv.w}, ba_[4] = {ba.x, ba.y, ba.z, ba.w};
            const float bv_[4] = {bv.x, bv.y, bv.z, bv.w}, la_[4] = {la.x, la.y, la.z, la.w};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const float pdd = sPdd[(t + q) * NV + j], pd = sPd[(t + q) * NV + j];
                a1 = fmaf(pdd, ra_[q], a1); a2 = fmaf(pd, rv_[q], a2);
                b1 = fmaf(pdd, ba_[q], b1); b2 = fmaf(pd, bv_[q], b2);
                if (!isx && t + q < NL) a3 = fmaf(sP[(t + q + 1) * NV + j], la_[q], a3);
            }
        }
        lam = (lam - a1) - a2;
        float lin = ((-lam - cb[lane]) - b1) - b2;
        if (!isx) {
            for (int i = 0; i < NL; i++) a3 = fmaf(-sP[(i + 1) * NV + j], LA[NL + i], a3);
            lin = lin - a3;
        }
        rhs[(isx ? 0 : 16) + j] = -lin;
    } else if (lane < 2 * NV + 3) rhs[NV + (lane - 2 * NV)] = bqx[lane - 2 * NV];
    else if (lane < 2 * NV + 7) rhs[16 + NV + (lane - 2 * NV - 3)] = bqy[lane - 2 * NV - 3];
    __syncwarp();
    if (lane < 2 * NV) {
        float acc = 0.0f;
        if (isx) {
#pragma unroll
            for (int k = 0; k < 14; k++) acc = fmaf(sKx[j * 14 + k], rhs[k], acc);
            a.cx[(size_t)g * NV + j] = acc;
        } else {
#pragma unroll
            for (int k = 0; k < 15; k++) acc = fmaf(sKy[j * 15 + k], rhs[16 + k], acc);
            a.cy[(size_t)g * NV + j] = acc;
        }
        cc[lane] = acc;
    }
    __syncwarp();
    // ---- trajectories of the projected coefficients  [projection.py:173-180]
#pragma unroll
    for (int k = 0; k < 2 * NV; k++) cr[k] = cc[k];
    for (int t = lane; t < T_; t += 32) {
        float xd, yd, xdd, ydd;
        dot11x2(sPd + t * NV, cr, xd, yd);
        dot11x2(sPdd + t * NV, cr, xdd, ydd);
        V0[t] = xd; V1[t] = yd; V2[t] = xdd; V3[t] = ydd;
        float acc = 0.0f;                         // y
#pragma unroll
        for (int k = 0; k < NV; k++) acc = fmaf(sP[t * NV + k], cr[NV + k], acc);
        V8[t] = acc;
    }
    __syncwarp();
    // ---- lane slack and residual  [projection.py:182-183]
    for (int i = lane; i < NL; i += 32) {
        float Ay = V8[i + 1];
        float s = dm::max0_(-Ay + c.b_lane_ub);
        sl[i] = s; LB[i] = (Ay - c.b_lane_ub) + s;
        Ay = -V8[i + 1];
        s = dm::max0_(-Ay + c.b_lane_lb);
        sl[NL + i] = s; LB[NL + i] = (Ay - c.b_lane_lb) + s;
    }
    // ---- compute_alph_d: polar step without unwrap, residuals  [projection.py:217-255]
    for (int t = lane; t < T_; t += 32) {
        float xd = V0[t], yd = V1[t], xdd = V2[t], ydd = V3[t];
        float bvx, bvy, bax, bay;
        polar_clip(dm::atan2_(yd, xd), xd, yd, c.v_min, c.v_max, bvx, bvy);
        polar_clip(dm::atan2_(ydd, xdd), xdd, ydd, 0.0f, c.a_max, bax, bay);
        V4[t] = xdd - bax; V5[t] = ydd - bay; V6[t] = xd - bvx; V7[t] = yd - bvy;
    }
    __syncwarp();
    // ---- residual norm in lane order  [projection.py:262-264]
    float res_norm;
    {
        float p = 0.0f;
        for (int t = lane; t < T_; t += 32) p = fmaf(V4[t], V4[t], p);
        for (int t = lane; t < T_; t += 32) p = fmaf(V5[t], V5[t], p);
        float n_acc = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_; t += 32) p = fmaf(V6[t], V6[t], p);
        for (int t = lane; t < T_; t += 32) p = fmaf(V7[t], V7[t], p);
        float n_vel = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int i = lane; i < 2 * NL; i += 32) p = fmaf(LB[i], LB[i], p);
        float n_lane = sqrtf(warp_sum(p));
        res_norm = (n_acc + n_vel) + n_lane;
    }
    // ---- multiplier update  [projection.py:267-272]
    if (lane < 2 * NV) {
        const float* rA = isx ? V4 : V5; const float* rV = isx ? V6 : V7;
        float a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
        for (int t = 0; t < T_; t += 4) {
            const float4 ra = *reinterpret_cast<const float4*>(rA + t), rv = *reinterpret_cast<const float4*>(rV + t);
            const float4 lb = *reinterpret_cast<const float4*>(LB + t);
            const float ra_[4] = {ra.x, ra.y, ra.z, ra.w}, rv_[4] = {rv.x, rv.y, rv.z, rv.w}, lb_[4] = {lb.x, lb.y, lb.z, lb.w};
#pragma unroll
            for (int q = 0; q < 4; q++) {
                a1 = fmaf(sPdd[(t + q) * NV + j], ra_[q], a1); a2 = fmaf(sPd[(t + q) * NV + j], rv_[q], a2);
                if (!isx && t + q < NL) a3 = fmaf(sP[(t + q + 1) * NV + j], lb_[q], a3);
            }
        }
        lam = (lam - a1) - a2;
        if (!isx) {
            for (int i = 0; i < NL; i++) a3 = fmaf(-sP[(i + 1) * NV + j], LB[NL + i], a3);
            lam = lam - a3;
        }
        ((isx ? a.lam_x : a.lam_y) + (size_t)g * NV)[j] = lam;
    }
    __syncwarp();
    // ---- controls  [cem_helper.py:540-551]   V4 = v, V5 = steer
    for (int t = lane; t < T_; t += 32) V4[t] = sqrtf(V0[t] * V0[t] + V1[t] * V1[t]);
    __syncwarp();
    float* accg = a.acc + (size_t)g * T_; float* steerg = a.steer + (size_t)g * T_;
    for (int t = lane; t < T_; t += 32) {
        float vn = (t + 1 < T_) ? V4[t + 1] : V4[T_ - 1];
        accg[t] = (vn - V4[t]) / c.dt;
        float xd = V0[t], yd = V1[t];
        float s2 = xd * xd + yd * yd;
        float curv = (V3[t] * xd - yd * V2[t]) / (s2 * sqrtf(s2));
        float st = dm::atan_(curv * c.wheel_base);
        V5[t] = st; steerg[t] = st;
    }
    __syncwarp();
    for (int t = lane; t < T_ - 1; t += 32) V6[t] = V5[t + 1] - V5[t];        // steering_vel
    __syncwarp();
    // ---- risk-independent cost terms in lane order  [cem_helper.py:232-262]
    {
        const float vdes = a.v_des[e];
        float p = 0.0f;
        for (int t = lane; t < T_; t += 32) { float d = V4[t] - vdes; p = fmaf(d, d, p); }
        float n_v = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_; t += 32) p = fmaf(V5[t], V5[t], p);
        float c_s = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_ - 1; t += 32) p = fmaf(V6[t], V6[t], p);
        float c_sv = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_ - 2; t += 32) { float d = V6[t + 1] - V6[t]; p = fmaf(d, d, p); }
        float c_sa = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_; t += 32) { float d = dm::max0_(fabsf(V5[t]) - c.steer_max); p = fmaf(d, d, p); }
        float p1 = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_ - 1; t += 32) { float d = dm::max0_(fabsf(V6[t]) - c.steer_rate_pen); p = fmaf(d, d, p); }
        float p2 = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_; t += 32) p = fmaf(V3[t], V3[t], p);
        float n_ydd = sqrtf(warp_sum(p));
        p = 0.0f;
        for (int t = lane; t < T_; t += 32) p = fmaf(V2[t], V2[t], p);
        float n_xdd = sqrtf(warp_sum(p));
        float base = ((((res_norm + 0.1f * n_v) + 0.1f * ((c_s + c_sv) + c_sa)) + 0.1f * (p1 + p2)) + 0.02f * n_ydd) + 0.02f * n_xdd;
        if (lane == 0) { a.res_norm[g] = res_norm; a.cost_base[g] = base; }
    }
}
