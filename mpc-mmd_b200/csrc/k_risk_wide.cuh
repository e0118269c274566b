// k_risk_wide.cuh -- cvar / saa / mmd_random with 65..1024 rollouts per CEM sample (num_reduced above MPCMMD_MAX_NR_DEV).
//
// The warp paths of k_rollouts (ROLL_FLY / ROLL_STAGED) rank and fold at most 64 per-rollout values per sample (rollout i = lane + 32 h).  Here
// a whole CTA owns one sample: its threads roll out the num_reduced rollouts with ROLL_FLY's rollout_risk (controls drawn inside the loop, the
// same noise paths and obstacle windows), keep the per-rollout (obstacle, lower lane, upper lane) maxima in shared memory and finish the risk
// functional CTA-wide.  The formulas are those of the warp paths and of the oracle (DESIGN.md section 3), generic in num_reduced:
//   cvar        the order statistics floor(q) / ceil(q) of q = alpha (nr - 1) in ascending NaN-last order (a bitonic sort of the three value
//               arrays at once), var = v_lo lw + v_hi hw, then the mean of the v[i] >= var as a sequential ascending-index float32 sum;
//   saa         the count of v > 0 (NaN does not count) over nr, from block counts;
//   mmd_random  beta = 1/nr, sigma = sigma_random: one ascending-j fma row chain per rollout, then the two ascending-i folds on one thread.
// Nothing depends on the CTA size: every result is a fixed-order chain or an exact count.
//
// k_noise_wide: the noise tables of one outer iteration for every episode of a solve, drawn at the start of that iteration (see enqueue_solve).
#pragma once
#include "k_risk.cuh"

#define WIDE_THREADS 256       // up to 4 rollouts per thread at num_reduced 1024; 3 CTAs per SM under WIDE_MAXNREG
// register cap of k_rollouts_wide: ptxas's own choice (64) spills 4..56 bytes in every instantiation (beta-table replay the most); a cap of 96
// leaves 58..72 registers and no spills, 3 CTAs of WIDE_THREADS per SM
#define WIDE_MAXNREG 96

// shared-memory layout (in 4-byte words): the three value arrays [3][nr], the sort keys [3][P] (P = the power of two >= nr; reused for the
// tail values of cvar and the row chains of mmd_random), the per-warp counts (<= 32) followed by cvar's six tail counts, and three scalars
struct WideLayout { int P, val, key, wcnt, res, total; };
__host__ __device__ inline WideLayout wide_layout(int nr) {
    WideLayout L;
    int P = 1; while (P < nr) P <<= 1;
    L.P = P; L.val = 0; L.key = (3 * nr + 3) & ~3; L.wcnt = L.key + 3 * P; L.res = L.wcnt + 40; L.total = L.res + 4;
    return L;
}

// order-preserving key: ascending float order with -0 == +0 and every NaN last (one key, 0xffffffff).  Costs are never -0 (they come out of
// max0_ / nmax_ from a +0 start), and the value read back at a rank only enters var = v_lo lw + v_hi hw, so which of two equal values a rank
// holds cannot change the result: any sort with this order gives the oracle's order statistics.
__device__ __forceinline__ uint32_t wide_key(float x) {
    const uint32_t u = dm::f2u(x + 0.0f);
    if (x != x) return 0xffffffffu;
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float wide_unkey(uint32_t k) {
    if (k == 0xffffffffu) return __int_as_float(0x7fffffff);
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

template <int NT, bool SORTED, int NZ>
__global__ void __maxnreg__(WIDE_MAXNREG) k_rollouts_wide(DCfg c, RiskArgs a) {
    extern __shared__ __align__(128) float sm[];
    const int g = blockIdx.x;
    if (g >= a.n_samples) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nr = c.nr, e = g / a.B;
    const WideLayout L = wide_layout(nr);
    float* val = sm + L.val;                         // [0][nr] obstacle, [1][nr] lower lane, [2][nr] upper lane
    int* wcnt = (int*)(sm + L.wcnt);
    float* res = sm + L.res;
#pragma unroll 1
    for (int r = tid; r < nr; r += NT) {
        float m, l, u;
        rollout_risk<true, SORTED, NZ>(c, a, g, e, r, nullptr, nullptr, a.state0 + e * 5, a.x_obs + (size_t)e * c.O * T_, a.y_obs + (size_t)e * c.O * T_, m, l, u);
        val[r] = m; val[nr + r] = l; val[2 * nr + r] = u;
    }
    __syncthreads();
    if (a.cost_kind == 1) {
        // ---- mmd_random  [cem.py:355-356, 404-424]: beta = 1/nr, sigma = sigma_random, lane = 0; row i's chains as mmd_cost_warp's
        float* tv = sm + L.key; float* uv = tv + nr;
        const float v = dm::kern_cost_v(c.kernel, c.sigma_random);
#pragma unroll 1
        for (int i = tid; i < nr; i += NT) {
            const float ci = val[i];
            float t = 0.0f;
#pragma unroll 1
            for (int j = 0; j < nr; j++) t = fmaf(dm::kern_cost(c.kernel, ci - val[j], v), c.beta_del, t);
            const float ei = dm::kern_cost(c.kernel, ci - 0.0f, v);
            float u = 0.0f;
#pragma unroll 1
            for (int j = 0; j < nr; j++) u = fmaf(ei, c.beta_del, u);
            tv[i] = t; uv[i] = u;
            a.beta[(size_t)g * nr + i] = c.beta_del;
        }
        __syncthreads();
        if (tid == 0) {
            float s1 = 0.0f, s2 = 0.0f;
#pragma unroll 1
            for (int i = 0; i < nr; i++) { s1 = fmaf(c.beta_del, tv[i], s1); s2 = fmaf(c.beta_del, uv[i], s2); }
            a.sigma[g] = c.sigma_random; a.risk[g] = c.ker_wt * (s1 - 2.0f * s2); a.lane[g] = 0.0f;
        }
    } else if (a.cost_kind == 2) {
        // ---- cvar  [costs.py:206-221, 137-158] of the three arrays
        const int P = L.P;
        uint32_t* key = (uint32_t*)(sm + L.key);
#pragma unroll 1
        for (int i = tid; i < 3 * P; i += NT) { const int k = i / P, j = i % P; key[i] = j < nr ? wide_key(val[k * nr + j]) : 0xffffffffu; }
        __syncthreads();
        // bitonic sort of the three key arrays, ascending (padding keys sort last, so ranks < nr hold the nr real keys)
#pragma unroll 1
        for (int size = 2; size <= P; size <<= 1) {
#pragma unroll 1
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
#pragma unroll 1
                for (int t = tid; t < 3 * (P >> 1); t += NT) {
                    const int k = t / (P >> 1), p = t % (P >> 1);
                    const int i = 2 * p - (p & (stride - 1)), j = i + stride;
                    uint32_t* kk = key + k * P;
                    const uint32_t x = kk[i], y = kk[j];
                    if ((x > y) == ((i & size) == 0)) { kk[i] = y; kk[j] = x; }
                }
                __syncthreads();
            }
        }
        const float q = c.alpha_quant * (float)(nr - 1);
        const float lo = floorf(q), hi = ceilf(q);
        const float hw = q - lo, lw = 1.0f - hw;
        int ilo = (int)lo, ihi = (int)hi;
        ilo = ilo < 0 ? 0 : (ilo > nr - 1 ? nr - 1 : ilo);
        ihi = ihi < 0 ? 0 : (ihi > nr - 1 ? nr - 1 : ihi);
        if (tid < 3) res[tid] = wide_unkey(key[tid * P + ilo]) * lw + wide_unkey(key[tid * P + ihi]) * hw;      // var of array tid
        __syncthreads();                                  // the key arrays become the tail buffers
        // tail of each array: n = #{i : v[i] >= var} by block counts; the nonzero tail values are compacted in index order and summed serially.
        // Skipping the zeros is exact: the sum starts at +0, and s + (+-0) == s for every s that can occur (+0 + -0 = +0 under round to nearest,
        // a nonzero or NaN s is unchanged).
        float* tail = sm + L.key;
        int* cnt = wcnt + NT / 32;                        // [3] tail counts, [3] nonzero tail values (block-uniform; kept in shared memory for the three summing warps)
#pragma unroll 1
        for (int k = 0; k < 3; k++) {
            const float* v = val + k * nr;
            const float vark = res[k];
            float* tk = tail + k * P;
            int n = 0, base = 0;
#pragma unroll 1
            for (int i0 = 0; i0 < nr; i0 += NT) {
                const int i = i0 + tid;
                const float vi = i < nr ? v[i] : 0.0f;
                const bool in = i < nr && vi >= vark, add = in && vi != 0.0f;
                const unsigned bal = __ballot_sync(FULL, add);
                if (lane == 0) wcnt[warp] = __popc(bal);
                n += __syncthreads_count(in);             // also orders the wcnt writes before the reads below
                int off = base, tot = 0;
#pragma unroll 1
                for (int w = 0; w < NT / 32; w++) { const int cw = wcnt[w]; off += w < warp ? cw : 0; tot += cw; }
                if (add) tk[off + __popc(bal & ((1u << lane) - 1u))] = vi;
                base += tot;
                __syncthreads();                          // wcnt is rewritten by the next chunk
            }
            if (tid == 0) { cnt[k] = n; cnt[3 + k] = base; }
        }
        __syncthreads();
        if (lane == 0 && warp < 3) {                      // one serial ascending-index sum per array, on three warps
            const int k = warp, nk = cnt[k], zk = cnt[3 + k];
            const float* tk = tail + k * P;
            float s = 0.0f;
#pragma unroll 1
            for (int i = 0; i < zk; i++) s = s + tk[i];
            res[k] = nk > 0 ? s / (float)nk : 0.0f;
        }
        __syncthreads();
        if (tid == 0) { a.risk[g] = res[0]; a.lane[g] = res[1] + res[2]; }
    } else {
        // ---- saa  [costs.py:223-234, 160-171]: the reference's float sums of ones are exact below 2^24, so they equal the integer counts
        int so = 0, sl = 0, su = 0;
#pragma unroll 1
        for (int i0 = 0; i0 < nr; i0 += NT) {
            const int i = i0 + tid;
            so += __syncthreads_count(i < nr && val[i] > 0.0f);
            sl += __syncthreads_count(i < nr && val[nr + i] > 0.0f);
            su += __syncthreads_count(i < nr && val[2 * nr + i] > 0.0f);
        }
        if (tid == 0) { a.risk[g] = (float)so / (float)nr; a.lane[g] = ((float)sl + (float)su) / (float)nr; }
    }
}

// noise tables of outer iteration `it` for episodes 0..n_ep-1 of a handle with num_reduced > MPCMMD_MAX_NR_DEV.  Such a handle holds z1 / z2 / z3,
// the beta keys and the Beta candidate table for ONE iteration per episode (episode stride, no iteration axis); z_cem keeps its [E][iters] slots.
// CTA b covers element chunk b % chunks of episode b / chunks, so no (episode, iteration) is left to a single CTA.  Every element is k_noise's
// per-element draw (same keys, same dr:: functions), so the tables are the same bits as k_noise's slot (e, it).
#define NOISE_WIDE_THREADS 256
__global__ void __launch_bounds__(NOISE_WIDE_THREADS) k_noise_wide(DCfg c, DWork w, int it, int chunks) {
    const int e = blockIdx.x / chunks, ch = blockIdx.x % chunks;
    const int n = c.nr * c.np, ncem = (c.B - c.n_el) * NPAR;
    dr::Key key; key.k0 = 0u; key.k1 = (uint32_t)(3 * w.idx_mpc[e] + 5 * it + 7);
    const dr::Key k1 = dr::split0(key), k2 = dr::split0(k1), k3 = dr::split0(k2);
    float* z1 = w.z1 + (size_t)e * n; float* z2 = w.z2 + (size_t)e * n; float* z3 = w.z3 + (size_t)e * n;
    float* zc = w.zcem + ((size_t)e * c.iters + it) * ncem;
    const int i0 = ch * NOISE_WIDE_THREADS + threadIdx.x, st = chunks * NOISE_WIDE_THREADS;
#pragma unroll 1
    for (int i = i0; i < n; i += st) {
        if (c.noise_kind == 0) {
            z1[i] = dr::normal_elem(k1, (uint32_t)n, (uint32_t)i);
            z2[i] = dr::normal_elem(k2, (uint32_t)n, (uint32_t)i);
        }
        z3[i] = dr::normal_elem(k3, (uint32_t)n, (uint32_t)i);
    }
#pragma unroll 1
    for (int i = i0; i < ncem; i += st) zc[i] = dr::normal_elem(k2, (uint32_t)ncem, (uint32_t)i);
    if (c.noise_kind == 1 && w.btab) {
        float* bt = w.btab + (size_t)e * (4 * GT_FIELDS) * n;
#pragma unroll 1
        for (int i = i0; i < 4 * n; i += st) {
            const int stream = i / n, el = i % n;
            dr::gamma_table_fill(dr::gamma_stream_key(k1, k2, stream), (uint32_t)n, (uint32_t)el, bt + (size_t)stream * GT_FIELDS * n + el);
        }
    }
    if (i0 == 0) {
        uint32_t* k = w.keys + (size_t)e * 4;
        k[0] = k1.k0; k[1] = k1.k1; k[2] = k2.k0; k[3] = k2.k1;
    }
}
// the emitted row's beta record (n_ep, nr): k_select copies it with its first SEL_THREADS threads, which covers num_reduced <= 64 only; solves
// of num_reduced > 64 copy the whole record of the last iteration's selection once, after it
__global__ void k_wide_beta_out(int nr, int B, int iters, const float* __restrict__ beta, const int32_t* __restrict__ o_sel, float* __restrict__ o_beta) {
    const int e = blockIdx.x;
    const size_t gs = (size_t)e * B + o_sel[(size_t)e * iters + iters - 1];
#pragma unroll 1
    for (int i = threadIdx.x; i < nr; i += blockDim.x) o_beta[(size_t)e * nr + i] = beta[gs * nr + i];
}
__host__ inline int noise_wide_chunks(const DCfg& d) {
    const long long n = (long long)d.nr * d.np, need = d.noise_kind == 1 ? 4 * n : n, ncem = (long long)(d.B - d.n_el) * NPAR;
    const long long m = need > ncem ? need : ncem;
    return (int)((m + NOISE_WIDE_THREADS - 1) / NOISE_WIDE_THREADS);
}
