// k_inner_big.cuh -- reduced-set inner CEM of mmd_opt for LARGE reduced sets (num_reduced 11 .. 40: BASELINE configs[3] sweeps {5, 10, 20, 40}).
// d = num_reduced^2 + 1 reaches 1601: the covariance alone is 10 MB per chain, so the chain state lives in a global (L2 / HBM) block instead of shared
// memory, num_reduced is a run-time value, and one CTA (256 or 1024 threads) walks the same phases as the generic shared-memory kernel (k_inner_cem, k_risk.cuh):
//   top-num_reduced |theta| per sample  ->  one task per (sample, reduced index) for the nm-term Laplace row sums (97 % of the exponentials)
//   ->  per-sample (nr+1) KKT solve  ->  stable rank-count selection  ->  covariance  ->  block-wide panel Cholesky (4 columns per panel, factor kept
//   transposed in the upper triangle)  ->  register-tiled multivariate-normal resampling  ->  risk of the chosen set.
// Same arithmetic contract as every other inner-CEM kernel (the oracle is generic in num_reduced); this path is the functional, bit-exact one --
// the tcgen05 blocked-Cholesky / MVN-GEMM formulation SURVEY.md section 7 (hard part 4) sketches would be a tolerance-parity variant and is not built.
// Replaces beta_cem.compute_cem (S/compute_beta.py:93-157) for nm + 1 > 101.
#pragma once
#include "k_risk.cuh"

#define BIG_THREADS 1024        // launches where every chain can have an SM to itself (<= one chain per SM); larger launches use BIG_THREADS_SMALL
#define BIG_THREADS_SMALL 256
struct BigLayout {          // per-chain global state in floats; offsets are multiples of 4
    size_t D, th, cost, betas, idxs, rs, key64, perm, C, mean, eth, xc, ecost, ebetas, eidxs, kscr, small, total;
    int ldc, kstride;
};
__host__ __device__ inline size_t al4z(size_t x) { return (x + 3) & ~(size_t)3; }
__host__ __device__ inline BigLayout big_layout(int nr, int S, int ne) {
    BigLayout L; const size_t nm = (size_t)nr * nr, d = nm + 1;
    L.ldc = (int)al4z(d);
    L.kstride = (int)al4z(2 * (size_t)nr * nr + 4 * (size_t)nr);          // per-sample scratch of the KKT stage: K, Lm (nr x nr each), rd, u, w, tv
    size_t q = 0;
    L.D = q; q += al4z(nm * nm);
    L.th = q; q += al4z((size_t)S * d); L.cost = q; q += al4z(S); L.betas = q; q += al4z((size_t)S * nr); L.idxs = q; q += al4z((size_t)S * nr);
    L.rs = q; q += al4z((size_t)S * nr); L.key64 = q; q += al4z(2 * (size_t)S); L.perm = q; q += al4z(S);
    L.C = q; q += d * (size_t)L.ldc; L.mean = q; q += al4z(d);
    L.eth = q; q += al4z((size_t)ne * d); L.xc = q; q += al4z((size_t)ne * d); L.ecost = q; q += al4z(ne); L.ebetas = q; q += al4z((size_t)ne * nr); L.eidxs = q; q += al4z((size_t)ne * nr);
    L.kscr = q; q += (size_t)S * L.kstride;
    L.small = q; q += 256;
    L.total = (q + 31) & ~(size_t)31;
    return L;
}

// top-nr |theta| of one row (stable, ascending), run-time nr: the insertion network of beta_topk with its state in memory
__device__ __forceinline__ void big_topk(const float* __restrict__ row, int nm, int nr, int* __restrict__ tv, int* __restrict__ ti) {
    for (int i = 0; i < nr; i++) { tv[i] = -1; ti[i] = -1; }
    for (int m = 0; m < nm; m++) {
        const int v = (int)(dm::f2u(row[m]) & 0x7fffffffu);
        if (v >= tv[0]) {
            tv[0] = v; ti[0] = m;
            for (int p = 0; p < nr - 1 && tv[p] >= tv[p + 1]; p++) {
                const int a = tv[p]; tv[p] = tv[p + 1]; tv[p + 1] = a;
                const int b = ti[p]; ti[p] = ti[p + 1]; ti[p + 1] = b;
            }
        }
    }
}
// the (nr+1) KKT solve and the cost of one beta sample; same operation order as beta_finish<NR> (k_risk.cuh), arrays in memory
template <int KER>
__device__ __forceinline__ float big_finish(const DCfg& c, int nr, int nm, const int* __restrict__ ti, float sigma, const float* __restrict__ rowsum,
                                            const float* __restrict__ D, float* __restrict__ beta, float* __restrict__ K, float* __restrict__ Lm,
                                            float* __restrict__ rd, float* __restrict__ u, float* __restrict__ w) {
    const dm::LapScale ls = dm::kern_scale<KER>(sigma);
    for (int i = 0; i < nr; i++) {
        K[i * nr + i] = 1.0f;
        for (int j = 0; j < i; j++) { const float k = dm::lap_(D[(size_t)ti[i] * nm + ti[j]], ls); K[i * nr + j] = k; K[j * nr + i] = k; }
    }
    for (int j = 0; j < nr; j++) {
        float acc = K[j * nr + j] + 0.05f;
        for (int k = 0; k < j; k++) acc = fmaf(-Lm[j * nr + k], Lm[j * nr + k], acc);
        const float dd = sqrtf(acc);
        Lm[j * nr + j] = dd; rd[j] = 1.0f / dd;
        for (int i = j + 1; i < nr; i++) {
            float aa = K[i * nr + j];
            for (int k = 0; k < j; k++) aa = fmaf(-Lm[i * nr + k], Lm[j * nr + k], aa);
            Lm[i * nr + j] = aa * rd[j];
        }
    }
    for (int i = 0; i < nr; i++) {
        float aa = c.inv_nm * rowsum[i], bb = 1.0f;
        for (int k = 0; k < i; k++) { aa = fmaf(-Lm[i * nr + k], u[k], aa); bb = fmaf(-Lm[i * nr + k], w[k], bb); }
        u[i] = aa * rd[i]; w[i] = bb * rd[i];
    }
    for (int i = nr - 1; i >= 0; i--) {
        float aa = u[i], bb = w[i];
        for (int k = i + 1; k < nr; k++) { aa = fmaf(-Lm[k * nr + i], u[k], aa); bb = fmaf(-Lm[k * nr + i], w[k], bb); }
        u[i] = aa * rd[i]; w[i] = bb * rd[i];
    }
    float su = 0.0f, sw = 0.0f;
    for (int i = 0; i < nr; i++) { su = su + u[i]; sw = sw + w[i]; }
    const float nu = (su - 1.0f) / sw;
    for (int i = 0; i < nr; i++) beta[i] = fmaf(-nu, w[i], u[i]);
    float s1 = 0.0f, s2 = 0.0f;
    for (int i = 0; i < nr; i++) {
        float t = 0.0f;
        for (int j = 0; j < nr; j++) t = fmaf(K[i * nr + j], beta[j], t);
        s1 = fmaf(beta[i], t, s1);
        s2 = fmaf(c.m2_inv_nm * rowsum[i], beta[i], s2);
    }
    return s1 + s2;
}

// one CTA per chain; chain g of this launch uses state block (g - g_base) (the host launches chain ranges that fit the scratch budget); KER: MMD kernel form
template <int NT, int KER = dm::KER_LAPLACE>
__global__ void __launch_bounds__(NT) k_inner_cem_big(DCfg c, RollArgs ra, float* __restrict__ state, int g_base, int n_chains) {
    __shared__ float blk[16];
    __shared__ float red[3 * MPCMMD_MAX_NR_DEV * (NT / 32)];
    const RiskArgs& a = ra.r;
    const int g = g_base + blockIdx.x;
    if (blockIdx.x >= n_chains || g >= a.n_samples) return;
    const int nr = c.nr, nm = c.nm, d = nm + 1, np = c.np, S = c.S_in, ne = c.n_el_in, e = g / a.B;
    const int tid = threadIdx.x, nt = NT, warp = tid >> 5, lane = tid & 31;
    const BigLayout L = big_layout(nr, S, ne);
    const int ldc = L.ldc;
    float* st = state + (size_t)blockIdx.x * L.total;
    float* D = st + L.D; float* th = st + L.th; float* cost = st + L.cost; float* betas = st + L.betas; int* idxs = (int*)(st + L.idxs);
    float* rs = st + L.rs; long long* key64 = (long long*)(st + L.key64); int* perm = (int*)(st + L.perm);
    float* C = st + L.C; float* mean = st + L.mean; float* eth = st + L.eth; float* xc = st + L.xc;
    float* ecost = st + L.ecost; float* ebetas = st + L.ebetas; int* eidxs = (int*)(st + L.eidxs); float* small = st + L.small;
    // ---- distance table of the mother features  [kernel_computation.py:31-33]
    const float* F = ra.feat + (size_t)g * nm * 2 * NV;
    for (size_t i = tid; i < (size_t)nm * nm; i += nt) {
        const float* Fa = F + (i / nm) * 2 * NV; const float* Fb = F + (i % nm) * 2 * NV;
        float dist = 0.0f;
#pragma unroll
        for (int f = 0; f < 2 * NV; f++) dist = dm::kern_dist_acc<KER>(dist, Fa[f], Fb[f]);
        D[i] = dist;
    }
    for (size_t i = tid; i < (size_t)S * d; i += nt) th[i] = __ldg(c.theta0 + i);
    __syncthreads();
    float* resb = a.res_beta + (size_t)g * c.iters_in;
    for (int it = 0; it < c.iters_in; it++) {
        const int s0 = it == 0 ? 0 : ne;
        // (A) top-nr per new sample, (B) row sums per (sample, reduced index), (C) KKT solve + cost per sample  [compute_beta.py:113-129, 70-91]
        for (int s = s0 + tid; s < S; s += nt) { float* ks = st + L.kscr + (size_t)s * L.kstride; big_topk(th + (size_t)s * d, nm, nr, (int*)(ks + 2 * nr * nr + 3 * nr), idxs + s * nr); }
        __syncthreads();
        for (int task = tid; task < (S - s0) * nr; task += nt) {
            const int s = s0 + task / nr, i = task % nr;
            rs[s * nr + i] = beta_rowsum<KER>(D, nm, idxs[s * nr + i], th[(size_t)s * d + nm]);
        }
        __syncthreads();
        for (int s = s0 + tid; s < S; s += nt) {
            float* ks = st + L.kscr + (size_t)s * L.kstride;
            cost[s] = big_finish<KER>(c, nr, nm, idxs + s * nr, th[(size_t)s * d + nm], rs + s * nr, D, betas + s * nr, ks, ks + nr * nr, ks + 2 * nr * nr,
                                 ks + 2 * nr * nr + nr, ks + 2 * nr * nr + 2 * nr);
        }
        __syncthreads();
        for (int s = tid; s < S; s += nt) key64[s] = sort_key64(cost[s], s);
        __syncthreads();
        for (int s = tid; s < S; s += nt) {            // stable argsort by rank counting; only the ne best are needed  [compute_beta.py:56]
            const long long ks = key64[s];
            int rank = 0;
            for (int j = 0; j < S; j++) rank += (key64[j] < ks) ? 1 : 0;
            if (rank < ne) perm[rank] = s;
        }
        __syncthreads();
        // elites (rank order), mean, centered rows  [compute_beta.py:56-61]
        for (int i = tid; i < ne * d; i += nt) eth[i] = th[(size_t)perm[i / d] * d + (i % d)];
        for (int i = tid; i < ne * nr; i += nt) { const int src = perm[i / nr] * nr + (i % nr); ebetas[i] = betas[src]; eidxs[i] = idxs[src]; }
        for (int i = tid; i < ne; i += nt) ecost[i] = cost[perm[i]];
        for (int i = tid; i < d; i += nt) {
            float s = 0.0f;
            for (int el = 0; el < ne; el++) s = s + th[(size_t)perm[el] * d + i];
            mean[i] = s / (float)ne;
        }
        __syncthreads();
        for (int i = tid; i < ne * d; i += nt) { const float v = eth[i]; th[i] = v; xc[i] = v - mean[i % d]; }
        for (int i = tid; i < ne * nr; i += nt) { betas[i] = ebetas[i]; idxs[i] = eidxs[i]; }
        for (int i = tid; i < ne; i += nt) cost[i] = ecost[i];
        __syncthreads();
        for (size_t i = tid; i < (size_t)d * d; i += nt) {      // jnp.cov (ddof = 1) + 0.05 I, lower triangle  [compute_beta.py:61]
            const int r = (int)(i / d), q = (int)(i % d);
            if (q <= r) {
                float acc = 0.0f;
                for (int el = 0; el < ne; el++) acc = fmaf(xc[(size_t)el * d + r], xc[(size_t)el * d + q], acc);
                acc = acc / (float)(ne - 1);
                if (r == q) acc = acc + 0.05f;
                C[(size_t)r * ldc + q] = acc;
            }
        }
        __syncthreads();
        // block-wide Cholesky, left-looking by panels of four columns, rows strided over the threads; entry (r, j) accumulates fma(-L_rk, L_jk, .) for k ascending,
        // then the pivot's sqrt / reciprocal scaling (the contract's order).  The factor is kept transposed in the upper triangle: LT[k][q] = L[q][k].
        // Two levels: at the start of every SUPER-PANEL of 16 columns one pass brings all 16 columns of every row up to date with the finished columns k < J0
        // (16 accumulators per row in registers: one load of L[r][k] feeds 16 fmas, the (nm+1)^2 factor streams from L2 once per 16 columns instead of once per 4);
        // the four 4-column panels inside then only add the columns k >= J0 of their own super-panel.  Per entry the k order stays ascending.
        for (int p = 0; p < (d + 3) / 4; p++) {
            const int j0 = 4 * p, J0 = j0 & ~15;
            if (j0 == J0 && J0 > 0) {
                for (int r = J0 + tid; r < d; r += nt) {
                    float acc[16];
                    float* crow = C + (size_t)r * ldc + J0;             // ldc is a multiple of 4 and J0 of 16: float4 accesses; columns beyond d stay inside the padded row only
                    const int nq = min(16, ldc - J0);                   // for the last, partial super-panel
#pragma unroll
                    for (int u = 0; u < 16; u += 4) {
                        if (u < nq) { const float4 v = *reinterpret_cast<const float4*>(crow + u); acc[u] = v.x; acc[u + 1] = v.y; acc[u + 2] = v.z; acc[u + 3] = v.w; }
                        else { acc[u] = 0.0f; acc[u + 1] = 0.0f; acc[u + 2] = 0.0f; acc[u + 3] = 0.0f; }
                    }
                    // L[r][k] is the one load per step that is private to the thread (L2 / HBM latency); the 16 column operands are the same for every thread
                    // (L1 hits).  J0 is a multiple of 16: the private loads are fetched eight steps ahead, double buffered.
                    const float* pr = C + r;
                    float cur[8], nxt[8];
#pragma unroll
                    for (int q = 0; q < 8; q++) cur[q] = pr[(size_t)q * ldc];
                    for (int k0 = 0; k0 < J0; k0 += 8) {
                        if (k0 + 8 < J0) {
#pragma unroll
                            for (int q = 0; q < 8; q++) nxt[q] = pr[(size_t)(k0 + 8 + q) * ldc];
                        }
#pragma unroll
                        for (int q = 0; q < 8; q++) {
                            const float lr = -cur[q];
                            const float* lrow = C + (size_t)(k0 + q) * ldc + J0;
#pragma unroll
                            for (int u = 0; u < 16; u += 4) {
                                if (u < nq) {
                                    const float4 l = *reinterpret_cast<const float4*>(lrow + u);
                                    acc[u] = fmaf(lr, l.x, acc[u]); acc[u + 1] = fmaf(lr, l.y, acc[u + 1]); acc[u + 2] = fmaf(lr, l.z, acc[u + 2]); acc[u + 3] = fmaf(lr, l.w, acc[u + 3]);
                                }
                            }
                        }
#pragma unroll
                        for (int q = 0; q < 8; q++) cur[q] = nxt[q];
                    }
#pragma unroll
                    for (int u = 0; u < 16; u += 4)
                        if (u < nq) *reinterpret_cast<float4*>(crow + u) = make_float4(acc[u], acc[u + 1], acc[u + 2], acc[u + 3]);
                }
                __syncthreads();
            }
            // every thread first finishes the partial sums of its rows, rows j0..j0+3 publish the diagonal block
            for (int r = j0 + tid; r < d; r += nt) {
                const float4 av = *reinterpret_cast<const float4*>(C + (size_t)r * ldc + j0);
                float a0 = av.x, a1 = av.y, a2 = av.z, a3 = av.w;
                for (int k = J0; k < j0; k++) {
                    const float lr = C[(size_t)k * ldc + r];
                    const float4 lj = *reinterpret_cast<const float4*>(C + (size_t)k * ldc + j0);
                    a0 = fmaf(-lr, lj.x, a0); a1 = fmaf(-lr, lj.y, a1); a2 = fmaf(-lr, lj.z, a2); a3 = fmaf(-lr, lj.w, a3);
                }
                *reinterpret_cast<float4*>(C + (size_t)r * ldc + j0) = make_float4(a0, a1, a2, a3);      // partial sums back in place (lower triangle)
                if (r < j0 + 4) { float* b = blk + 4 * (r - j0); b[0] = a0; b[1] = a1; b[2] = a2; b[3] = a3; }
            }
            __syncthreads();
            const float b00 = blk[0], b10 = blk[4], b11 = blk[5], b20 = blk[8], b21 = blk[9], b22 = blk[10];
            const float b30 = blk[12], b31 = blk[13], b32 = blk[14], b33 = blk[15];
            const float d0 = sqrtf(b00), r0 = 1.0f / d0;
            const float l10 = b10 * r0, l20 = b20 * r0, l30 = b30 * r0;
            const float d1 = sqrtf(fmaf(-l10, l10, b11)), r1 = 1.0f / d1;
            const float l21 = fmaf(-l20, l10, b21) * r1, l31 = fmaf(-l30, l10, b31) * r1;
            const float d2 = sqrtf(fmaf(-l21, l21, fmaf(-l20, l20, b22))), r2 = 1.0f / d2;
            const float l32 = fmaf(-l31, l21, fmaf(-l30, l20, b32)) * r2;
            const float d3 = sqrtf(fmaf(-l32, l32, fmaf(-l31, l31, fmaf(-l30, l30, b33)))), r3 = 1.0f / d3;
            for (int r = j0 + tid; r < d; r += nt) {
                const float4 av = *reinterpret_cast<const float4*>(C + (size_t)r * ldc + j0);
                float a0 = av.x, a1 = av.y, a2 = av.z, a3 = av.w;
                float e0 = a0 * r0;
                a1 = fmaf(-e0, l10, a1); float e1 = a1 * r1;
                a2 = fmaf(-e1, l21, fmaf(-e0, l20, a2)); float e2 = a2 * r2;
                a3 = fmaf(-e2, l32, fmaf(-e1, l31, fmaf(-e0, l30, a3))); float e3 = a3 * r3;
                if (r == j0) e0 = d0;
                if (r == j0 + 1) e1 = d1;
                if (r == j0 + 2) e2 = d2;
                if (r == j0 + 3) e3 = d3;
                if (r >= j0 + 0) C[(size_t)(j0 + 0) * ldc + r] = e0;
                if (r >= j0 + 1 && j0 + 1 < d) C[(size_t)(j0 + 1) * ldc + r] = e1;
                if (r >= j0 + 2 && j0 + 2 < d) C[(size_t)(j0 + 2) * ldc + r] = e2;
                if (r >= j0 + 3 && j0 + 3 < d) C[(size_t)(j0 + 3) * ldc + r] = e3;
            }
            __syncthreads();
        }
        // resample  [compute_beta.py:63-66]: task = (new row r, 8 consecutive columns); acc_u = sum_{k <= q0+u} L[q0+u][k] z[r][k], k ascending
        {
            const int nrow = S - ne;
            const float* zT = c.zb_iterT + (size_t)it * d * nrow;
            const int NQ8 = (d + 7) / 8;
            for (int task = tid; task < NQ8 * nrow; task += nt) {
                const int q0 = 8 * (task / nrow), r = task % nrow;
                float acc[8];
#pragma unroll
                for (int u = 0; u < 8; u++) acc[u] = 0.0f;
                const float* zp = zT + r;
                for (int k = 0; k <= q0; k++) {
                    const float z = __ldg(zp + (size_t)k * nrow);
                    const float* Ck = C + (size_t)k * ldc + q0;
#pragma unroll
                    for (int u = 0; u < 8; u++) if (q0 + u < d) acc[u] = fmaf(Ck[u], z, acc[u]);
                }
#pragma unroll
                for (int kk = 1; kk < 8; kk++) {
                    const int k = q0 + kk;
                    if (k < d) {
                        const float z = __ldg(zp + (size_t)k * nrow);
#pragma unroll
                        for (int u = kk; u < 8; u++) if (q0 + u < d) acc[u] = fmaf(C[(size_t)k * ldc + q0 + u], z, acc[u]);
                    }
                }
                float* dst = th + (size_t)(ne + r) * d + q0;
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
                for (int i = 0; i < nr; i++) { small[i] = ebetas[i]; ((int*)small)[64 + i] = eidxs[i]; }
                small[200] = th[(size_t)perm[0] * d + nm];
            }
        }
        __syncthreads();
    }
    // ---- risk of the chosen reduced set (its rollouts come back from global memory)  [costs.py:173-186, 121-135]
    const int* ridx = (const int*)small + 64;
    const float* xg = ra.xroll + (size_t)g * nm * np; const float* yg = ra.yroll + (size_t)g * nm * np;
    const float* xo = a.x_obs + (size_t)e * c.O * T_; const float* yo = a.y_obs + (size_t)e * c.O * T_;
    constexpr int NW = NT / 32;
    for (int r = 0; r < nr; r++) {
        const float* xred = xg + (size_t)ridx[r] * np; const float* yred = yg + (size_t)ridx[r] * np;
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
        float cs[MPCMMD_MAX_NR_DEV], lbv[MPCMMD_MAX_NR_DEV], ubv[MPCMMD_MAX_NR_DEV], beta[MPCMMD_MAX_NR_DEV];
        for (int r = 0; r < nr; r++) {
            float m = red[(r * 3 + 0) * NW], l = red[(r * 3 + 1) * NW], u = red[(r * 3 + 2) * NW];
            for (int wv = 1; wv < NW; wv++) { m = dm::nmax_(m, red[(r * 3 + 0) * NW + wv]); l = dm::nmax_(l, red[(r * 3 + 1) * NW + wv]); u = dm::nmax_(u, red[(r * 3 + 2) * NW + wv]); }
            cs[r] = m; lbv[r] = l; ubv[r] = u; beta[r] = small[r];
            a.beta[(size_t)g * nr + r] = small[r];
        }
        const float sigma = small[200];
        a.sigma[g] = sigma;
        a.risk[g] = mmd_cost<KER>(c, beta, cs, sigma);
        a.lane[g] = mmd_cost<KER>(c, beta, lbv, sigma) + mmd_cost<KER>(c, beta, ubv, sigma);
    }
}
