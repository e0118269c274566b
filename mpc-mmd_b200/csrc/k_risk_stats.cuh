// k_risk_stats.cuh -- per-plan Monte-Carlo risk statistics of the per-rollout costs (DESIGN.md section 3 item 9): collision and lane
// probabilities, mean, VaR / CVaR (the solver's cvar_cost formula in float64) and the Laplace-kernel MMD of the obstacle cost.
//
// One CTA per plan.  The CTA
//   1. counts the lane hits (c_lane > 0 or NaN);
//   2. counts the obstacle hits and NaNs, and compacts the positive obstacle costs as uint64 bit patterns (a non-negative double orders
//      like its bits) into the plan's c_lane row, with the eight 8-bit digit histograms on the side.  The zeros are the head of the
//      sorted order, so only the positive costs are sorted; the order of the compaction does not matter, the sorted sequence is unique;
//   3. LSD radix-sorts the compacted keys between the c_lane and c_obs rows (stable in-tile ranks from __match_any_sync, per-warp digit
//      counts scanned over warps in order); a pass whose digit is the same for every key is skipped;
//   4. reduces over the sorted keys in a fixed order: the mean, VaR at alpha * (n - 1) (__dmul_rn / __dadd_rn: no contraction), the CVaR
//      suffix, and for the MMD E = sum exp(-c / sigma) and the all-pairs sum S = n + 2 sum_i P_i, P_{i+1} = (P_i + 1) exp(-(v_{i+1} - v_i) / sigma),
//      as a scan of the affine maps P -> d P + d: each thread composes its contiguous segment, the segments combine in a fixed tree.
// Every result depends only on the multiset of a plan's costs, so it is the same at any chunking.  c_obs and c_lane are overwritten.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define RS_THREADS 512
#define RS_WARPS (RS_THREADS / 32)
#define RS_OUT 6                 // per plan: p_coll, p_lane, mean_obs, var_obs, cvar_obs, mmd_obs

// the composite of the maps of a run of sorted values: P_last = a P_in + b, sum of the run's P = cs P_in + ds
struct RsAffine { double a, b, cs, ds; };
__device__ __forceinline__ RsAffine rs_combine(const RsAffine& l, const RsAffine& r) {      // l first, then r
    RsAffine o;
    o.a = r.a * l.a; o.b = r.a * l.b + r.b;
    o.cs = l.cs + r.cs * l.a; o.ds = l.ds + r.cs * l.b + r.ds;
    return o;
}

__device__ __forceinline__ double rs_warp_sum(double v) {
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    return v;
}
// fixed-order block sum (every thread gets the result); red: RS_WARPS doubles
__device__ __forceinline__ double rs_block_sum(double v, double* red) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    v = rs_warp_sum(v);
    __syncthreads();
    if (lane == 0) red[w] = v;
    __syncthreads();
    double t = lane < RS_WARPS ? red[lane] : 0.0;
    return rs_warp_sum(t);
}
__device__ __forceinline__ unsigned rs_block_count(unsigned v, unsigned* cnt) {
    for (int off = 16; off >= 1; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
    __syncthreads();
    if (threadIdx.x == 0) *cnt = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(cnt, v);
    __syncthreads();
    return *cnt;
}
__device__ __forceinline__ void rs_shfl_affine(RsAffine& x, int off) {
    RsAffine r;
    r.a = __shfl_down_sync(0xffffffffu, x.a, off); r.b = __shfl_down_sync(0xffffffffu, x.b, off);
    r.cs = __shfl_down_sync(0xffffffffu, x.cs, off); r.ds = __shfl_down_sync(0xffffffffu, x.ds, off);
    if (((threadIdx.x & 31) & (2 * off - 1)) == 0) x = rs_combine(x, r);
}

// grid = plans of this chunk.  c_obs, c_lane (gridDim.x, n), overwritten; sigma (gridDim.x,) or null (no MMD); out (gridDim.x, RS_OUT).
__global__ void __launch_bounds__(RS_THREADS) k_risk_stats(int n, double alpha, double ker_wt, const double* __restrict__ sigma,
                                                           double* __restrict__ c_obs, double* __restrict__ c_lane, double* __restrict__ out) {
    __shared__ unsigned s_hist[8][256];
    __shared__ unsigned s_wcnt[RS_WARPS][256];   // per-tile digit counts of each warp (zero between tiles)
    __shared__ unsigned s_woff[RS_WARPS][256];   // their scanned offsets
    __shared__ unsigned s_base[256];
    __shared__ unsigned s_cnt[4];                // compacted count, block counters
    __shared__ double s_red[RS_WARPS];
    __shared__ RsAffine s_aff[RS_WARPS];
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const size_t off = (size_t)blockIdx.x * n;
    const double* lrow = c_lane + off;
    const double* orow = c_obs + off;
    unsigned long long* buf0 = reinterpret_cast<unsigned long long*>(c_lane + off);
    unsigned long long* buf1 = reinterpret_cast<unsigned long long*>(c_obs + off);
    for (int i = tid; i < 8 * 256; i += RS_THREADS) (&s_hist[0][0])[i] = 0;
    for (int i = tid; i < RS_WARPS * 256; i += RS_THREADS) (&s_wcnt[0][0])[i] = 0;
    if (tid == 0) s_cnt[0] = 0;

    // ---- 1. lane hits
    unsigned hl = 0;
    const unsigned un = (unsigned)n;
    for (unsigned i = tid; i < un; i += RS_THREADS) { const double v = lrow[i]; hl += (v > 0.0) || (v != v); }
    const unsigned hits_lane = rs_block_count(hl, &s_cnt[1]);        // (its barriers also order step 1's reads before step 2's writes)

    // ---- 2. obstacle hits, NaNs, compaction of the positive costs into buf0 (the c_lane row) + digit histograms
    unsigned ho = 0, hn = 0;
    const unsigned lt = (1u << lane) - 1u;
    for (unsigned base = 0; base < un; base += RS_THREADS) {
        const unsigned i = base + tid;
        const double v = i < un ? orow[i] : 0.0;
        const bool nan = v != v, pos = v > 0.0;
        ho += pos || nan; hn += nan;
        const unsigned m = __ballot_sync(0xffffffffu, pos);
        unsigned b = 0;
        if (lane == 0 && m) b = atomicAdd(&s_cnt[0], __popc(m));
        b = __shfl_sync(0xffffffffu, b, 0);
        if (pos) {
            const unsigned long long k = (unsigned long long)__double_as_longlong(v);
            buf0[b + __popc(m & lt)] = k;
#pragma unroll
            for (int p = 0; p < 8; p++) atomicAdd(&s_hist[p][(k >> (8 * p)) & 255u], 1u);
        }
    }
    const unsigned hits_obs = rs_block_count(ho, &s_cnt[2]);
    const unsigned nans = rs_block_count(hn, &s_cnt[3]);
    const unsigned m = s_cnt[0];                                     // positive costs; the other n - m are 0 (or NaN)
    double* o = out + (size_t)blockIdx.x * RS_OUT;
    if (tid == 0) { o[0] = (double)hits_obs / (double)n; o[1] = (double)hits_lane / (double)n; }
    const double sg = sigma ? sigma[blockIdx.x] : 0.0;
    if (nans) {                                                      // NumPy semantics: any NaN makes every moment NaN
        if (tid == 0) { const double q = __longlong_as_double(0x7ff8000000000000LL); o[2] = q; o[3] = q; o[4] = q; o[5] = sigma ? q : 0.0; }
        return;
    }

    // ---- 3. LSD radix sort of buf0[0, m)
    unsigned long long *src = buf0, *dst = buf1;
    for (int p = 0; p < 8 && m > 1; p++) {
        if (__syncthreads_or(tid < 256 && s_hist[p][tid] == m)) continue;       // every key has this digit: the pass is the identity
        if (w == 0) {                                                           // exclusive scan of the digit histogram
            unsigned c[8], t = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) { c[k] = s_hist[p][lane * 8 + k]; t += c[k]; }
            unsigned incl = t;
            for (int d = 1; d < 32; d <<= 1) { const unsigned u = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += u; }
            unsigned run = incl - t;
#pragma unroll
            for (int k = 0; k < 8; k++) { s_base[lane * 8 + k] = run; run += c[k]; }
        }
        const int sh = 8 * p;
        for (unsigned t0 = 0; t0 < m; t0 += RS_THREADS) {
            const unsigned i = t0 + tid;
            const bool valid = i < m;
            const unsigned long long k = valid ? src[i] : 0ull;
            const unsigned d = valid ? (unsigned)((k >> sh) & 255u) : 256u;
            const unsigned peers = __match_any_sync(0xffffffffu, d);
            const unsigned rank = __popc(peers & lt);
            if (valid && rank == 0) s_wcnt[w][d] = __popc(peers);
            __syncthreads();
            if (tid < 256) {                                                    // digit tid: offsets of the warps in order, counts re-zeroed
                unsigned run = s_base[tid];
                for (int x = 0; x < RS_WARPS; x++) { const unsigned cx = s_wcnt[x][tid]; s_woff[x][tid] = run; run += cx; s_wcnt[x][tid] = 0; }
                s_base[tid] = run;
            }
            __syncthreads();
            if (valid) dst[s_woff[w][d] + rank] = k;
        }
        __syncthreads();
        unsigned long long* t = src; src = dst; dst = t;
    }
    __syncthreads();
    const double* s = reinterpret_cast<const double*>(src);          // the positive costs, ascending
    const size_t z = (size_t)n - m;                                  // zeros ahead of them

    // ---- 4. statistics
    double acc = 0.0;
    for (unsigned j = tid; j < m; j += RS_THREADS) acc += s[j];
    const double sum_all = rs_block_sum(acc, s_red);
    const double q = __dmul_rn(alpha, (double)(n - 1));
    const double lo = floor(q), hi = ceil(q);
    const double hw = __dadd_rn(q, -lo), lw = __dadd_rn(1.0, -hw);
    const size_t ilo = (size_t)lo, ihi = (size_t)hi;
    const double vlo = ilo < z ? 0.0 : s[ilo - z], vhi = ihi < z ? 0.0 : s[ihi - z];
    const double var = __dadd_rn(__dmul_rn(vlo, lw), __dmul_rn(vhi, hw));
    // CVaR: the costs >= var are all n when var == 0, else the sorted suffix from the first s[j] >= var
    unsigned j0 = 0;
    if (var > 0.0) {
        unsigned a = 0, b = m;                                       // binary search (uniform over the CTA)
        while (a < b) { const unsigned mid = (a + b) >> 1; if (s[mid] >= var) b = mid; else a = mid + 1; }
        j0 = a;
    }
    double cs = 0.0;
    if (var > 0.0) for (unsigned j = j0 + tid; j < m; j += RS_THREADS) cs += s[j];
    const double sum_tail = var > 0.0 ? rs_block_sum(cs, s_red) : sum_all;
    const double n_tail = var > 0.0 ? (double)(m - j0) : (double)n;
    double mmd = 0.0;
    if (sigma) {
        double e = 0.0;
        for (unsigned j = tid; j < m; j += RS_THREADS) e += exp(-s[j] / sg);
        const double E = (double)z + rs_block_sum(e, s_red);
        // thread tid's contiguous segment of the sorted positive costs
        const unsigned j1 = (unsigned)(((unsigned long long)m * tid) / RS_THREADS), j2 = (unsigned)(((unsigned long long)m * (tid + 1)) / RS_THREADS);
        RsAffine f = {1.0, 0.0, 0.0, 0.0};
        double prev = j1 > 0 ? s[j1 - 1] : (z > 0 ? 0.0 : (m > 0 ? s[0] : 0.0));
        for (unsigned j = j1; j < j2; j++) {
            const double d = exp(-(s[j] - prev) / sg);
            prev = s[j];
            f.a = f.a * d; f.b = (f.b + 1.0) * d;
            f.cs = f.cs + f.a; f.ds = f.ds + f.b;
        }
        for (int x = 1; x < 32; x <<= 1) rs_shfl_affine(f, x);
        __syncthreads();
        if (lane == 0) s_aff[w] = f;
        __syncthreads();
        if (w == 0) {
            f = lane < RS_WARPS ? s_aff[lane] : RsAffine{1.0, 0.0, 0.0, 0.0};
            for (int x = 1; x < 32; x <<= 1) rs_shfl_affine(f, x);
            if (lane == 0) {
                // the z zeros first (d = 1: P_i = P_in + i), from P_in = -1 so that the first value gets P = 0
                const double zd = (double)z;
                const RsAffine head = {1.0, zd, zd, 0.5 * zd * (zd + 1.0)};
                const RsAffine all = rs_combine(head, f);
                const double sp = -all.cs + all.ds;
                const double S = (double)n + 2.0 * sp, nd = (double)n;
                mmd = ker_wt * (S / (nd * nd) - 2.0 * E / nd);
            }
        }
    }
    if (tid == 0) { o[2] = sum_all / (double)n; o[3] = var; o[4] = sum_tail / n_tail; o[5] = mmd; }
}
