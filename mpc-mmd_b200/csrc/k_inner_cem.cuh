// k_inner_cem.cuh -- the reduced-set inner CEM of mmd_opt for num_reduced^2 + 1 <= 32 (num_reduced <= 5), the dominant
// kernel of a solve.  Same arithmetic contract as the generic kernel (k_risk.cuh) and oracle_inner_cem (bit for bit), but
// mapped for instruction issue, which is what bounds it (DESIGN.md 5.3 / 5.4: its time follows its executed instructions):
//   * Laplace kernel entries k(d; sigma) = 2^(-(d s2)) (DESIGN.md 3.4) two at a time on Blackwell's packed FP32 pipe (FFMA2 / FADD2 / FMUL2,
//     IEEE per lane), four columns of a distance row per 16-byte shared-memory load,
//   * top-(num_reduced + 1) |theta| selection on packed (value | index) integer keys by a min / max merge network (exact path on near ties),
//   * elite selection by ONE warp with redux.sync min over per-lane sorted candidate lists (no O(S^2) rank count),
//   * covariance (exact division by num_elite - 1 = 10), panel Cholesky by one warp (one range check per pivot: dm::sqrt_rcp) and the
//     multivariate-normal resampling in packed FP32 with float4 shared-memory operands,
//   * the reference's sample / elite counts (100 / 11) as template constants, so the shared-memory layout folds into immediate offsets.
// Latency builds (k_inner_cem_lat, the LAT build of k_inner_cem_fast) spread a chain over up to 16 warps and factor in registers (icl_chol_regs).
// Replaces beta_cem.compute_cem (S/compute_beta.py:93-157) + kernel_matrix.compute_kernel (S/kernel_computation.py:19-65)
// + Costs.compute_mmd_obs / compute_mmd_lane (S/optimizer/costs.py:121-135, 173-186).
#pragma once
#include <type_traits>
#include "k_risk.cuh"

namespace pk {   // packed float32x2 arithmetic (sm_100a): each lane is an IEEE-754 round-to-nearest operation
typedef unsigned long long f2;
__device__ __forceinline__ f2 pack(float lo, float hi) { f2 r; asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ f2 dup(float v) { return pack(v, v); }
__device__ __forceinline__ void unpack(f2 v, float& lo, float& hi) { asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ float lo(f2 v) { float a, b; unpack(v, a, b); return a; }
__device__ __forceinline__ float hi(f2 v) { float a, b; unpack(v, a, b); return b; }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { f2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f2 add2(f2 a, f2 b) { f2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f2 mul2(f2 a, f2 b) { f2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
// 16-byte shared-memory load from a 32-bit shared-window address (volatile: stays inside its loop trip, in program order with the barriers around the phase)
__device__ __forceinline__ uint32_t smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float4 lds128(uint32_t a) {
    float4 v; asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a)); return v;
}
// MUFU.EX2 (opt-in fast-math mode only, MPCMMD_MATH=fast): 2^x to ~2^-22 relative, not reproducible on the CPU oracle
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
}  // namespace pk

// Laplace kernel entries k(d; sigma) two at a time (dm::lap_ per lane, operation for operation).  LapK carries the per-bandwidth constants: exact contract
// (FM = false): sc2 = (-s2, -s2) and the distance cap; fast math (FM = true): sc2 = -s2 in both lanes, the exponentials run on the XU pipe (MUFU.EX2).
// KER = kernel form (dm::KER_*): the Gaussian entry is the same function of a stored squared distance with its own scale g2 in place of s2 (dm::kern_scale).
struct LapK { pk::f2 sc2; float dcap; };
template <bool FM, int KER = dm::KER_LAPLACE>
__device__ __forceinline__ LapK lap_k(float sigma) {
    LapK k;
    if constexpr (FM) { k.sc2 = pk::dup(dm::kern_ns2<KER>(sigma)); k.dcap = 0.0f; }
    else { const dm::LapScale L = dm::kern_scale<KER>(sigma); k.sc2 = pk::dup(L.ns2); k.dcap = L.dcap; }
    return k;
}
namespace pk {
// two dm::lap_ at once.  The clamp is a scalar instruction whose destination is free, so it drops each distance straight into the register pair the packed
// polynomial works on; the 2^n scaling stays a float multiply (a NaN distance or bandwidth stays a NaN).
__device__ __forceinline__ f2 lap2_exact(float da, float db, f2 ns2, float dcap) {
    const float MAGIC = 12582912.0f;
    float sa, sb;
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(sa) : "f"(da), "f"(dcap));
    asm("min.NaN.f32 %0, %1, %2;" : "=f"(sb) : "f"(db), "f"(dcap));
    const f2 dc = pack(sa, sb);
    const f2 t = fma2(dc, ns2, dup(MAGIC));
    const f2 f = fma2(dc, ns2, fma2(t, dup(-1.0f), dup(MAGIC)));          // MAGIC - t is exact
    f2 p = dup(DM_LAP_C6);
    p = fma2(p, f, dup(DM_LAP_C5)); p = fma2(p, f, dup(DM_LAP_C4)); p = fma2(p, f, dup(DM_LAP_C3));
    p = fma2(p, f, dup(DM_LAP_C2)); p = fma2(p, f, dup(DM_LAP_C1)); p = fma2(p, f, dup(1.0f));
    float ta, tb; unpack(t, ta, tb);
    // bits(t) = bits(MAGIC) + n and bits(MAGIC) << 23 == 0 (mod 2^32)  =>  (bits(t) << 23) + 0x3f800000 = bits(2^n)
    const float sca = dm::u2f((dm::f2u(ta) << 23) + 0x3f800000u), scb = dm::u2f((dm::f2u(tb) << 23) + 0x3f800000u);
    return mul2(p, pack(sca, scb));
}
}  // namespace pk
template <bool FM>
__device__ __forceinline__ pk::f2 lap2(float da, float db, const LapK& k) {
    if constexpr (FM) { float a, b; pk::unpack(pk::mul2(pk::pack(da, db), k.sc2), a, b); return pk::pack(pk::ex2_approx(a), pk::ex2_approx(b)); }
    else return pk::lap2_exact(da, db, k.sc2, k.dcap);
}

#define ICF_THREADS 96
#define ICF_MAX_S 128       // candidates per inner iteration handled by the one-warp selection (4 per lane)
#define ICF_MAX_NE 12       // elites (covariance operands are read as 3 float4 per column)

struct FastLayout {         // shared-memory carve-up in floats; every offset is a multiple of 4 floats
    int D, th, cost, betas, idxs, eth, ecost, ebetas, eidxs, perm, xc, C, mean, small, red, total;
    int ldt, ldc, ldd;
};
__host__ __device__ inline FastLayout fast_layout(int nr, int S, int ne) {
    FastLayout L; const int nm = nr * nr, d = nm + 1;
    L.ldt = d | 1;                           // odd row stride: thread-per-row accesses are bank-conflict free
    L.ldc = al4(d);
    L.ldd = al4(nm);                         // distance-table row stride: rows start 16-byte aligned, so the row-sum loop reads four columns per LDS.128
    int q = 0;
    L.D = q; q += nm * L.ldd;
    {   // the S - ne resampled rows (iteration 0: the first S - ne rows of the constant theta0 table; the rest sit in the elite buffer); the region is also borrowed by the
        // mother features while D is built and by the centered elites xc between the elite gather and the covariance (the rows are dead then)
        int n = (S - ne) * L.ldt;
        if (nm * 2 * NV > n) n = nm * 2 * NV;
        if (ICF_MAX_NE * L.ldc > n) n = ICF_MAX_NE * L.ldc;
        L.th = q; L.xc = q; q += al4(n);
    }
    L.cost = q; L.betas = q; L.idxs = q;                 // cost: see C below      // the per-row beta / packed-index records live in a global scratch (L2): only <= ne of S rows are read back
                                                           // per iteration, and the 2.4 KB they took in shared memory is what separates 9 from 10 chains per SM
    L.eth = q; q += al4(ne * L.ldt); L.ecost = q; q += al4(ne); L.ebetas = q; q += al4(ne * nr); L.eidxs = q; q += al4(ne);      // single buffers: readers finish before a barrier, writers start after it
    L.perm = q; q += al4(ne);
    L.C = q; L.cost = q; q += d * L.ldc;     // covariance (lower, row-major); overwritten in place by L transposed (LT[k][q] = L[q][k]).  The S sample
                                             // costs borrow the same region: they live from the evaluation to the selection, C from the covariance to the resampling
    L.mean = q; q += L.ldc;
    L.small = q; q += 52; L.red = q;
    L.total = q;
    return L;
}

// exact top-NR |theta| (stable, ascending) -- used when the packed keys below cannot decide
template <int NR>
__device__ __noinline__ int top_abs_exact(const float* __restrict__ row) {     // returns the indices packed 5 bits each
    constexpr int nm = NR * NR;
    int tv[NR], ti[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) { tv[i] = -1; ti[i] = -1; }
#pragma unroll 1
    for (int m = 0; m < nm; m++) {
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
    int packed = 0;
#pragma unroll
    for (int i = 0; i < NR; i++) packed |= ti[i] << (5 * i);
    return packed;
}

// the QP + MMD cost of one beta sample given its reduced set (indices ti, ascending |theta|) and bandwidth sigma
// [compute_beta.py:70-91, 120-129]; bit-identical to the second half of beta_sample<NR> of k_risk.cuh
// LDD = row stride of D in floats; a multiple of four selects the vectorised row-sum loop (four columns per 16-byte load, same operations in the same order)
template <int NR, bool FM = false, int LDD = NR * NR, int KER = dm::KER_LAPLACE>
__device__ __forceinline__ float beta_eval(const DCfg& c, const int (&ti)[NR], float sigma, const float* __restrict__ D,
                                           float* __restrict__ beta_out, int* __restrict__ idx_out /* one packed word */) {
    constexpr int nm = NR * NR;
    constexpr bool VEC = (LDD % 4 == 0) && nm >= 4;
    constexpr int MV = VEC ? (nm & ~3) : 0;          // columns handled by the vectorised loop
    const LapK rinv2 = lap_k<FM, KER>(sigma);
    // ---- ker_mixed row sums: rowsum_i = sum_m k(D[idx_i][m]; sigma), ascending m  [kernel_computation.py:31-37, compute_beta.py:77]
    constexpr int NP = NR / 2;                       // pairs of reduced rows handled together
    pk::f2 rs2[NP > 0 ? NP : 1];
    float rsl = 0.0f;                                // last row when NR is odd
#pragma unroll
    for (int p = 0; p < NP; p++) rs2[p] = pk::dup(0.0f);
    const float* Dr[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) Dr[i] = D + ti[i] * LDD;       // D is symmetric bit for bit: row idx_i
    if constexpr (VEC) {
        // Addresses: one loop-carried register (table base + 4 m) and one multiply-add per row and trip, instead of an index and a scaled add per row.
        uint32_t dmo = pk::smem_addr(D);
#pragma unroll 1
        for (int m = 0; m < MV; m += 4, dmo += 16) {
#pragma unroll
            for (int p = 0; p < NP; p++) {
                const float4 va = pk::lds128(dmo + (uint32_t)ti[2 * p] * (LDD * 4)), vb = pk::lds128(dmo + (uint32_t)ti[2 * p + 1] * (LDD * 4));
                rs2[p] = pk::add2(rs2[p], lap2<FM>(va.x, vb.x, rinv2));
                rs2[p] = pk::add2(rs2[p], lap2<FM>(va.y, vb.y, rinv2));
                rs2[p] = pk::add2(rs2[p], lap2<FM>(va.z, vb.z, rinv2));
                rs2[p] = pk::add2(rs2[p], lap2<FM>(va.w, vb.w, rinv2));
            }
            if constexpr (NR & 1) {
                const float4 vc = pk::lds128(dmo + (uint32_t)ti[NR - 1] * (LDD * 4));
                pk::f2 e = lap2<FM>(vc.x, vc.y, rinv2);
                rsl = rsl + pk::lo(e); rsl = rsl + pk::hi(e);
                e = lap2<FM>(vc.z, vc.w, rinv2);
                rsl = rsl + pk::lo(e); rsl = rsl + pk::hi(e);
            }
        }
    }
#pragma unroll 1
    for (int m = MV; m + 1 < nm; m += 2) {
#pragma unroll
        for (int p = 0; p < NP; p++) {
            rs2[p] = pk::add2(rs2[p], lap2<FM>(Dr[2 * p][m], Dr[2 * p + 1][m], rinv2));
            rs2[p] = pk::add2(rs2[p], lap2<FM>(Dr[2 * p][m + 1], Dr[2 * p + 1][m + 1], rinv2));
        }
        if constexpr (NR & 1) {
            const pk::f2 e = lap2<FM>(Dr[NR - 1][m], Dr[NR - 1][m + 1], rinv2);
            rsl = rsl + pk::lo(e); rsl = rsl + pk::hi(e);
        }
    }
    if constexpr (nm & 1) {                          // last column
        constexpr int m = nm - 1;
#pragma unroll
        for (int p = 0; p < NP; p++) rs2[p] = pk::add2(rs2[p], lap2<FM>(Dr[2 * p][m], Dr[2 * p + 1][m], rinv2));
        if constexpr (NR & 1) rsl = rsl + pk::lo(lap2<FM>(Dr[NR - 1][m], Dr[NR - 1][m], rinv2));
    }
    float rowsum[NR];
#pragma unroll
    for (int p = 0; p < NP; p++) pk::unpack(rs2[p], rowsum[2 * p], rowsum[2 * p + 1]);
    if constexpr (NR & 1) rowsum[NR - 1] = rsl;
    // ---- ker_red (symmetric bit for bit); diagonal k(0) = 1
    float K[NR][NR];
    {
        constexpr int NE = NR * (NR - 1) / 2;
        float dv[NE + 1];
        int e = 0;
#pragma unroll
        for (int i = 0; i < NR; i++) {
            K[i][i] = 1.0f;
#pragma unroll
            for (int j = 0; j < i; j++) dv[e++] = Dr[i][ti[j]];
        }
        dv[NE] = dv[NE - 1];
        float ev[NE + 1];
#pragma unroll
        for (int q = 0; q < NE; q += 2) pk::unpack(lap2<FM>(dv[q], dv[q + 1], rinv2), ev[q], ev[q + 1]);
        e = 0;
#pragma unroll
        for (int i = 0; i < NR; i++)
#pragma unroll
            for (int j = 0; j < i; j++) { K[i][j] = ev[e]; K[j][i] = ev[e]; e++; }
    }
    // ---- A = ker_red + 0.05 I, Cholesky with reciprocal pivots; the two right-hand sides (kbar, 1) are solved as one packed pair
    float Lm[NR][NR], rd[NR];
#pragma unroll
    for (int j = 0; j < NR; j++) {
        float acc = K[j][j] + 0.05f;
#pragma unroll
        for (int k = 0; k < j; k++) acc = fmaf(-Lm[j][k], Lm[j][k], acc);
        float dd; dm::sqrt_rcp(acc, dd, rd[j]);
        Lm[j][j] = dd;
#pragma unroll
        for (int i = j + 1; i < NR; i++) {
            float aa = K[i][j];
#pragma unroll
            for (int k = 0; k < j; k++) aa = fmaf(-Lm[i][k], Lm[j][k], aa);
            Lm[i][j] = aa * rd[j];
        }
    }
    pk::f2 uw[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) {
        pk::f2 ab = pk::pack(c.inv_nm * rowsum[i], 1.0f);
#pragma unroll
        for (int k = 0; k < i; k++) ab = pk::fma2(pk::dup(-Lm[i][k]), uw[k], ab);
        uw[i] = pk::mul2(ab, pk::dup(rd[i]));
    }
#pragma unroll
    for (int i = NR - 1; i >= 0; i--) {
        pk::f2 ab = uw[i];
#pragma unroll
        for (int k = i + 1; k < NR; k++) ab = pk::fma2(pk::dup(-Lm[k][i]), uw[k], ab);
        uw[i] = pk::mul2(ab, pk::dup(rd[i]));
    }
    float u[NR], w[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) pk::unpack(uw[i], u[i], w[i]);
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
    int packed = 0;
#pragma unroll
    for (int i = 0; i < NR; i++) packed |= ti[i] << (5 * i);
    *idx_out = packed;
    return s1 + s2;
}

// one beta sample of the inner CEM [compute_beta.py:113-129, 70-91]; bit-identical to beta_sample<NR> of k_risk.cuh
template <int NR, bool FM = false, int LDD = NR * NR, int KER = dm::KER_LAPLACE>
__device__ __forceinline__ float beta_sample_fast(const DCfg& c, const float* __restrict__ row, const float* __restrict__ D,
                                                  float* __restrict__ beta_out, int* __restrict__ idx_out /* one packed word */) {
    constexpr int nm = NR * NR;
    static_assert(nm <= 32, "index must fit in the 5 low key bits");
    // ---- top-NR |theta|: keys (|theta| bits with the 5 low bits replaced by the index) kept as the NR+1 largest, ascending.
    // Key order equals the (|theta|, index) order of jnp.argsort unless two entries share their upper 26 value bits; the
    // (NR+1)-th key is kept so that such a near tie at the boundary is seen too.
    int tk[NR + 1];
#pragma unroll
    for (int p = 0; p <= NR; p++) tk[p] = 0;
    auto insert = [&](float x, int m) {
        const int v = (int)((dm::f2u(x) & 0x7fffffe0u) | (uint32_t)m);
        tk[0] = max(tk[0], v);
#pragma unroll
        for (int p = 0; p < NR; p++) { const int lo = min(tk[p], tk[p + 1]), hi = max(tk[p], tk[p + 1]); tk[p] = lo; tk[p + 1] = hi; }
    };
    if constexpr (NR == 5) {
        // four keys at a time: sort them (5 exchanges), keep the six largest of {list, group} with the half-cleaner c_i = max(t_i, s_(3-i)) (the list has six entries,
        // the group four: t_4, t_5 pass), and sort the resulting bitonic sequence with the 7-exchange merger (0,4)(1,5) (0,2)(1,3) (0,1)(2,3)(4,5) (minimal for the
        // reachable 0-1 patterns, found by search): 28 min / max operations per four keys instead of 44 by insertion.  The keys are distinct (index bits), so the sorted
        // list is the same list.
#define ICF_CE(a, b) { const int lo_ = min(a, b), hi_ = max(a, b); a = lo_; b = hi_; }
#pragma unroll 1
        for (int m = 0; m + 3 < nm; m += 4) {        // rolled: the whole kernel's loop body has to stay inside the 32 KB instruction cache
            int s0 = (int)((dm::f2u(row[m]) & 0x7fffffe0u) | (uint32_t)m), s1 = (int)((dm::f2u(row[m + 1]) & 0x7fffffe0u) | (uint32_t)(m + 1));
            int s2 = (int)((dm::f2u(row[m + 2]) & 0x7fffffe0u) | (uint32_t)(m + 2)), s3 = (int)((dm::f2u(row[m + 3]) & 0x7fffffe0u) | (uint32_t)(m + 3));
            ICF_CE(s0, s1) ICF_CE(s2, s3) ICF_CE(s0, s2) ICF_CE(s1, s3) ICF_CE(s1, s2)
            tk[0] = max(tk[0], s3); tk[1] = max(tk[1], s2); tk[2] = max(tk[2], s1); tk[3] = max(tk[3], s0);
            ICF_CE(tk[0], tk[4]) ICF_CE(tk[1], tk[5]) ICF_CE(tk[0], tk[2]) ICF_CE(tk[1], tk[3]) ICF_CE(tk[0], tk[1]) ICF_CE(tk[2], tk[3]) ICF_CE(tk[4], tk[5])
        }
#undef ICF_CE
#pragma unroll
        for (int m = nm & ~3; m < nm; m++) insert(row[m], m);
    } else {
#pragma unroll NR
        for (int m = 0; m < nm; m++) insert(row[m], m);      // partially unrolled (instruction cache, see above)
    }
    int ti[NR];
    bool near = false;
#pragma unroll
    for (int p = 0; p < NR; p++) { ti[p] = tk[p + 1] & 31; near |= ((tk[p] ^ tk[p + 1]) < 32); }
    if (near) {
        const int pkd = top_abs_exact<NR>(row);
#pragma unroll
        for (int p = 0; p < NR; p++) ti[p] = (pkd >> (5 * p)) & 31;
    }
    return beta_eval<NR, FM, LDD, KER>(c, ti, row[nm], D, beta_out, idx_out);
}

// float -> uint32 whose unsigned order is "ascending float, -0 == +0, NaN last" (jnp.argsort order of the costs)
__device__ __forceinline__ uint32_t sort_key32(float x) {
    const float xz = x + 0.0f;
    const uint32_t u = dm::f2u(xz);
    uint32_t k = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    if (xz != xz) k = 0xffffffffu;
    return k;
}


// stable argsort of the S candidate costs, first ne entries, by ONE warp (S <= 128): candidate j < n_old is elite j (cost ecost[j]),
// else new row j - n_old (cost[j - n_old]).  Each lane sorts its four candidates (j = lane + 32u, stable), then ne rounds of
// redux.sync min pick the globally smallest (key, index).  Writes perm[0..ne) and the winners' costs.  [compute_beta.py:56]
// (ecost_n may be the same buffer as ecost: every read of the old elite costs precedes the first write)
__device__ __forceinline__ void icf_select(int lane, int S, int n_old, int ne, const float* ecost, const float* __restrict__ cost, int* __restrict__ perm, float* ecost_n) {
    uint32_t k0, k1, k2, k3; int j0, j1, j2, j3;
    {
        uint32_t kk[4]; int jj[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            const int j = lane + 32 * u;
            if (j < S) { kk[u] = sort_key32(j < n_old ? ecost[j] : cost[j - n_old]); jj[u] = j; }
            else { kk[u] = 0xffffffffu; jj[u] = 0x7fffffff; }
        }
        // stable local sort (adjacent exchanges only; indices ascend within a lane)
#define ICF_CE(x, y) { const bool sw_ = kk[y] < kk[x]; const uint32_t ka_ = kk[x], kb_ = kk[y]; const int ja_ = jj[x], jb_ = jj[y]; \
                       kk[x] = sw_ ? kb_ : ka_; kk[y] = sw_ ? ka_ : kb_; jj[x] = sw_ ? jb_ : ja_; jj[y] = sw_ ? ja_ : jb_; }
        ICF_CE(0, 1) ICF_CE(1, 2) ICF_CE(2, 3) ICF_CE(0, 1) ICF_CE(1, 2) ICF_CE(0, 1)
#undef ICF_CE
        k0 = kk[0]; k1 = kk[1]; k2 = kk[2]; k3 = kk[3]; j0 = jj[0]; j1 = jj[1]; j2 = jj[2]; j3 = jj[3];
    }
    int mine = 0;
#pragma unroll 1
    for (int r = 0; r < ne; r++) {
        const uint32_t m = __reduce_min_sync(FULL, k0);
        const uint32_t wj = __reduce_min_sync(FULL, (k0 == m) ? (uint32_t)j0 : 0x7fffffffu);
        if ((uint32_t)j0 == wj) { k0 = k1; k1 = k2; k2 = k3; k3 = 0xffffffffu; j0 = j1; j1 = j2; j2 = j3; j3 = 0x7fffffff; }
        if (lane == r) mine = (int)wj;
    }
    float won = 0.0f;
    if (lane < ne) won = mine < n_old ? ecost[mine] : cost[mine - n_old];
    __syncwarp();                                  // every read of the old elite costs precedes the overwrite (one buffer)
    if (lane < ne) { perm[lane] = mine; ecost_n[lane] = won; }
}

// Cholesky of the d x d covariance by ONE warp, left-looking by PANELS of four columns: lane r owns row r.  For panel j0 = 4p each lane first
// accumulates its four entries (r, j0..j0+3) over the finished columns k < j0 -- four independent fma chains per lane, two FFMA2, that share one load
// of L[r][k] and the broadcast L[j0..j0+3][k] (the factor is kept TRANSPOSED: LT[k][q] = L[q][k], so both are conflict-free) -- then the
// 4 x 4 diagonal block is gathered with ten shuffles and factored REDUNDANTLY by every lane in registers (no exchange inside the panel): the lanes of
// the block store their row of it, the lanes below finish their own four entries with the block's columns and store them transposed.  The last
// panel factors only the columns that exist (d = 26: two).  Entry (r, j) accumulates fma(-L_rk, L_jk, .) for k = 0 .. j-1 ascending, then
// the pivot's square root / reciprocal scaling: the contract's order, bit for bit the same as the column-by-column versions.  In place: LT lives in
// the upper triangle (and diagonal) of C while the untouched part of C's lower triangle still holds the covariance.  The resampling loops read
// whole float4 groups from the diagonal's group on (icf_mvn_row_unrolled, icf_mvn_row_regs), so the only zero fill they need is the strict lower
// triangle of each 4 x 4 diagonal block (LT[k][q] = 0 for 4 (k / 4) <= q < k); the rest of the lower triangle is never read again.
// One panel of W <= 4 live columns j0 .. j0 + W - 1 (W < 4 only for the last panel of a d that is not a multiple of four).
template <int d, int W, bool LAST>
__device__ __forceinline__ void icf_chol_panel_step(float* __restrict__ C, const float* __restrict__ rowp, int r, int lane, int p) {
    constexpr int ldc = (d + 3) & ~3;
    const int j0 = 4 * p;
    float a[4];
    {
        // a(r, j0..j0+3), then the k < j0 part on the packed pipe: each lane of an FFMA2 is the fma(-L_rk, L_jk, .) of one entry, k ascending
        pk::f2 a01 = *reinterpret_cast<const pk::f2*>(rowp + j0), a23 = *reinterpret_cast<const pk::f2*>(rowp + j0 + 2);
        const float* pr = C + r;                                       // LT[k][r] = L[r][k], k = 0, 1, ...
        const float* pj = C + j0;                                      // L[j0..j0+3][k]
#pragma unroll 1
        for (int k4 = 0; k4 < p; k4++) {                               // j0 is a multiple of four: whole groups of four columns, fixed offsets
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const pk::f2 nl = pk::dup(-pr[u * ldc]);
                if constexpr (W > 2) {
                    const pk::f2 l01 = *reinterpret_cast<const pk::f2*>(pj + u * ldc), l23 = *reinterpret_cast<const pk::f2*>(pj + u * ldc + 2);
                    a01 = pk::fma2(nl, l01, a01); a23 = pk::fma2(nl, l23, a23);
                } else {
                    const float2 lj = *reinterpret_cast<const float2*>(pj + u * ldc);
                    a01 = pk::fma2(nl, pk::pack(lj.x, lj.y), a01);
                }
            }
            pr += 4 * ldc; pj += 4 * ldc;
        }
        pk::unpack(a01, a[0], a[1]); pk::unpack(a23, a[2], a[3]);
    }
    // diagonal block b(i, j), j <= i < W, from lanes j0 + i, factored redundantly by every lane (the columns that exist only).  The pivots take the
    // branch-free fast path of sqrt_rcp with one range check for the whole block; the block is the same on every lane, so is the check, and a block
    // with a pivot outside the fast path's range is factored again with sqrt_rcp -- the same bits either way.
    float b[4][4], l[4][4], dv[4], rv[4];
#pragma unroll
    for (int i = 0; i < W; i++)
#pragma unroll
        for (int j = 0; j <= i; j++) b[i][j] = __shfl_sync(FULL, a[j], j0 + i);
    auto factor = [&](auto fast) {
        bool ok = true;
#pragma unroll
        for (int j = 0; j < W; j++) {
            float acc = b[j][j];
#pragma unroll
            for (int k = 0; k < j; k++) acc = fmaf(-l[j][k], l[j][k], acc);
            if constexpr (decltype(fast)::value) ok &= dm::sqrt_rcp_fast(acc, dv[j], rv[j]);
            else dm::sqrt_rcp(acc, dv[j], rv[j]);
#pragma unroll
            for (int i = j + 1; i < W; i++) {
                float s = b[i][j];
#pragma unroll
                for (int k = 0; k < j; k++) s = fmaf(-l[i][k], l[j][k], s);
                l[i][j] = s * rv[j];
            }
        }
        return ok;
    };
    if (!factor(std::true_type{})) factor(std::false_type{});
    if (lane >= j0 && lane < j0 + W) {
        // row v = lane - j0 of the block of LT: zeros left of the diagonal, the pivot, then L[j0 + u][j0 + v] = l[u][v] (the padding columns of the last panel get zeros)
        const int v = lane - j0;
        float o[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            float x = 0.0f;
            if (u < W) {
                x = u == W - 1 ? dv[u] : 0.0f;                     // v <= W - 1: the last column needs no test for its pivot
#pragma unroll
                for (int w = 0; w < u; w++) x = v == w ? l[u][w] : x;
                if (u < W - 1) x = v == u ? dv[u] : x;
            }
            o[u] = x;
        }
        *reinterpret_cast<float4*>(C + lane * ldc + j0) = make_float4(o[0], o[1], o[2], o[3]);
    }
    if constexpr (!LAST) {
        // rows below the block: own entries L[r][j0 + u], stored transposed as column r of LT rows j0..j0+3
        float e[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
            float s = a[u];
#pragma unroll
            for (int k = 0; k < u; k++) s = fmaf(-e[k], l[u][k], s);
            e[u] = s * rv[u];
        }
        if (lane >= j0 + 4 && lane < d) {
#pragma unroll
            for (int u = 0; u < 4; u++) C[(j0 + u) * ldc + lane] = e[u];
        }
    }
    __syncwarp();                                                  // the next panel (or the caller) reads these rows of LT
}
template <int d>
__device__ __forceinline__ void icf_chol_panel(float* __restrict__ C, int ldc_, int lane) {
    constexpr int NG = (d + 3) / 4, ldc = (d + 3) & ~3;    // the row stride is a compile-time constant (every caller passes al4(d)): immediate load offsets
    (void)ldc_;
    const int r = lane < d ? lane : d - 1;                 // lanes >= d shadow the last row (no stores)
    const float* rowp = C + r * ldc;
#pragma unroll 1
    for (int p = 0; p < NG - 1; p++) icf_chol_panel_step<d, 4, false>(C, rowp, r, lane, p);
    icf_chol_panel_step<d, d - 4 * (NG - 1), true>(C, rowp, r, lane, NG - 1);
}

// one covariance task: C[r][4*q4 .. 4*q4+3] = (sum_el xc[el][r] * xc[el][q]) / (ne - 1) (+ 0.05 on the diagonal), el ascending  [compute_beta.py:61]
__device__ __forceinline__ void icf_cov_task(const float* __restrict__ xc, float* __restrict__ C, int ldc, int ne, int r, int q4) {
    const float nm1 = (float)(ne - 1);
    pk::f2 a01 = pk::dup(0.0f), a23 = pk::dup(0.0f);
#pragma unroll
    for (int el = 0; el < ICF_MAX_NE; el++) {
        if (el < ne) {
            const float xr = xc[el * ldc + r];
            const float4 xq = *reinterpret_cast<const float4*>(xc + el * ldc + 4 * q4);
            a01 = pk::fma2(pk::dup(xr), pk::pack(xq.x, xq.y), a01);
            a23 = pk::fma2(pk::dup(xr), pk::pack(xq.z, xq.w), a23);
        }
    }
    float o[4]; pk::unpack(a01, o[0], o[1]); pk::unpack(a23, o[2], o[3]);
#pragma unroll
    for (int u = 0; u < 4; u++) { o[u] = (ne == 11) ? dm::div10(o[u]) : o[u] / nm1; if (4 * q4 + u == r) o[u] = o[u] + 0.05f; }
    *reinterpret_cast<float4*>(C + r * ldc + 4 * q4) = make_float4(o[0], o[1], o[2], o[3]);
}

// one resampled row: acc[p] = (sum_k L[2p][k] z[k], sum_k L[2p+1][k] z[k]), k ascending  [compute_beta.py:63].  LT[k][q] = 0 for q < k, so a
// term with k > q adds an exact zero and whole float4 groups can be used.  Fully unrolled over k with the exact triangular group sets: ~40 % fewer
// executed instructions than a rolled k loop for ~450 more of code (the CTA-per-chain kernel's warps run in near lockstep and share the instruction cache)
template <int d>
__device__ __forceinline__ void icf_mvn_row_unrolled(const float* __restrict__ LT, int ldc, const float* __restrict__ zT, int nrow, int r, pk::f2 (&acc)[2 * ((d + 3) / 4)]) {
    constexpr int NG = (d + 3) / 4;
#pragma unroll
    for (int p = 0; p < 2 * NG; p++) acc[p] = pk::dup(0.0f);
#pragma unroll
    for (int k = 0; k < d; k++) {
        const pk::f2 z2 = pk::dup(__ldg(zT + k * nrow + r));
#pragma unroll
        for (int g4 = k / 4; g4 < NG; g4++) {
            const float4 l = *reinterpret_cast<const float4*>(LT + k * ldc + 4 * g4);
            acc[2 * g4] = pk::fma2(pk::pack(l.x, l.y), z2, acc[2 * g4]);
            acc[2 * g4 + 1] = pk::fma2(pk::pack(l.z, l.w), z2, acc[2 * g4 + 1]);
        }
    }
}

// the same row with the d normals already in registers (latency build: they are fetched before the one-warp Cholesky, whose duration hides
// their L2 latency; with one chain per SM nothing else would)
template <int d>
__device__ __forceinline__ void icf_mvn_row_regs(const float* __restrict__ LT, int ldc, const float (&z)[d], pk::f2 (&acc)[2 * ((d + 3) / 4)]) {
    constexpr int NG = (d + 3) / 4;
#pragma unroll
    for (int p = 0; p < 2 * NG; p++) acc[p] = pk::dup(0.0f);
#pragma unroll
    for (int k = 0; k < d; k++) {
        const pk::f2 z2 = pk::dup(z[k]);
#pragma unroll
        for (int g4 = k / 4; g4 < NG; g4++) {
            const float4 l = *reinterpret_cast<const float4*>(LT + k * ldc + 4 * g4);
            acc[2 * g4] = pk::fma2(pk::pack(l.x, l.y), z2, acc[2 * g4]);
            acc[2 * g4 + 1] = pk::fma2(pk::pack(l.z, l.w), z2, acc[2 * g4 + 1]);
        }
    }
}

template <int d> __device__ __forceinline__ void icl_chol_regs(float* __restrict__ C, int lane);
// LAT = the build for launches that fit in a single wave of CTAs (one episode = 100 chains): no register cap (156 instead of the 56 registers
// that let 12 chains share an SM) and the resampling normals prefetched behind the Cholesky (mmd_opt p50 at batch 1: 8.3 -> 7.4 ms)
// FM = opt-in fast-math build (MPCMMD_MATH=fast): the Laplace-kernel exponentials on MUFU.EX2 instead of the contract's polynomial; tolerance parity only
// SC / NEC = compile-time copies of the inner CEM's sample / elite counts (0 = read them from the configuration): with the reference's sizes (100 / 11) baked in, the
// whole shared-memory layout folds into immediate offsets, which takes the address arithmetic the 56-register cap otherwise re-derives in every phase out of the kernel
// KER = MMD kernel form (dm::KER_*): changes only the distance table and the per-bandwidth scale
template <int NR, bool LAT, bool FM = false, int SC = 0, int NEC = 0, int KER = dm::KER_LAPLACE>
__global__ void __launch_bounds__(ICF_THREADS, LAT ? 3 : 12) k_inner_cem_fast(DCfg c, RollArgs ra) {
    extern __shared__ __align__(128) float sm[];
    const RiskArgs& a = ra.r;
    const int g = blockIdx.x;
    if (g >= a.n_samples) return;
    constexpr int nm = NR * NR, d = nm + 1, LDD = (nm + 3) & ~3;       // = FastLayout::ldd
    static_assert(d <= 32, "one covariance row per lane");
    constexpr int NPAIR = (d + 1) / 2;               // packed column pairs of a covariance / Cholesky row
    const int tid = threadIdx.x, nt = ICF_THREADS, warp = tid >> 5, lane = tid & 31;
    const int S = SC ? SC : c.S_in, ne = NEC ? NEC : c.n_el_in;
    const FastLayout L = fast_layout(NR, S, ne);
    const int ldt = L.ldt, ldc = L.ldc;
    float* D = sm + L.D; float* th = sm + L.th; float* cost = sm + L.cost; float* betas = ra.bscratch + (size_t)g * S * (NR + 1); int* idxs = (int*)(betas + S * NR);
    int* perm = (int*)(sm + L.perm); float* xc = sm + L.xc; float* C = sm + L.C; float* LT = C; float* mean = sm + L.mean;
    float* small = sm + L.small;
    float* eth = sm + L.eth;
    float* ecost = sm + L.ecost; float* eb = sm + L.ebetas; int* ei = (int*)(sm + L.eidxs);
    // ---- distance table of the mother features  [kernel_computation.py:31-33]; the features borrow the th region
    {
        float* F = th;
        const float* Fg = ra.feat + (size_t)g * nm * 2 * NV;
#pragma unroll 1
        for (int i = tid; i < nm * 2 * NV; i += nt) F[i] = Fg[i];
        __syncthreads();
#pragma unroll 1
        for (int i = tid; i < nm * nm; i += nt) {
            const float* Fa = F + (i / nm) * 2 * NV; const float* Fb = F + (i % nm) * 2 * NV;
            float dist = 0.0f;
#pragma unroll 2
            for (int f = 0; f < 2 * NV; f++) dist = dm::kern_dist_acc<KER>(dist, Fa[f], Fb[f]);
            D[(i / nm) * LDD + i % nm] = dist;
        }
        __syncthreads();
    }
    // ---- iteration 0 evaluates the S rows of theta0, later iterations the S - ne resampled rows.  theta0 (a constant table) is staged in shared memory once: its first
    //      S - ne rows into the row region, the last ne into the elite buffer (no elites exist before the first selection), so every iteration reads its rows with
    //      shared-memory loads at a compile-time stride -- new row s lives at th[s] for s < S - ne, else at eth[s - (S - ne)] (only iteration 0 has such rows)
    // covariance task of this thread: row cr, columns 4*cg .. 4*cg+3 (lower triangle in groups of four; tasks beyond nt wrap)
    int cr = -1, cg = 0, cr2 = -1, cg2 = 0;
    {
        int t = 0;
#pragma unroll 1
        for (int r = 0; r < d; r++) {
#pragma unroll 1
            for (int q4 = 0; q4 <= r / 4; q4++) { if (t == tid) { cr = r; cg = q4; } if (t == tid + nt) { cr2 = r; cg2 = q4; } t++; }
        }
    }
    {
        const int nrow0 = S - ne;
#pragma unroll 1
        for (int i = tid; i < S * d; i += nt) {
            const int s0 = i / d, q = i - s0 * d;
            (s0 < nrow0 ? th + s0 * ldt : eth + (s0 - nrow0) * ldt)[q] = c.theta0[i];
        }
    }
    __syncthreads();
    float* resb = a.res_beta + (size_t)g * c.iters_in;
#pragma unroll 1
    for (int it = 0; it < c.iters_in; it++) {
        const int n_old = it == 0 ? 0 : ne, n_new = S - n_old;
        const int nrow = S - ne;
        // -- evaluate the new rows (the elites keep last iteration's cost: same row => same arithmetic => same bits)
#pragma unroll 1
        for (int s = tid; s < n_new; s += nt) cost[s] = beta_sample_fast<NR, FM, LDD, KER>(c, s < nrow ? th + s * ldt : eth + (s - nrow) * ldt, D, betas + s * NR, idxs + s);
        __syncthreads();
        // -- stable argsort, first ne entries: candidate j < n_old is elite j, else new row j - n_old  [compute_beta.py:56]
        if (warp == 0) icf_select(lane, S, n_old, ne, ecost, cost, perm, ecost);
        __syncthreads();
        // -- gather the elites (rank order), their mean and the centered rows  [compute_beta.py:56-61].  Two phases around a barrier: every
        //    read of the old elite rows / the new rows happens before any write, so the elites need one buffer and xc can live in the (now
        //    dead) row region
        float v[ICF_MAX_NE]; float mu = 0.0f, gb = 0.0f; int gi = 0;
        if (tid < d) {
            float s = 0.0f;
#pragma unroll
            for (int el = 0; el < ICF_MAX_NE; el++) {
                if (el < ne) {
                    const int p = perm[el];
                    const int pn = p - n_old;          // new row index; rows beyond the row region exist in iteration 0 only (staged in the elite buffer)
                    v[el] = (p < n_old ? eth + p * ldt : pn < nrow ? th + pn * ldt : eth + (pn - nrow) * ldt)[tid];
                    s = s + v[el];
                }
            }
            mu = s / (float)ne;
        } else if (tid >= 32 && tid - 32 < ne * NR) {           // one (elite, component) per thread: ne * NR <= 64
            const int i = tid - 32, p = perm[i / NR], k = i % NR;
            gb = p < n_old ? eb[p * NR + k] : betas[(p - n_old) * NR + k];
            if (i < ne) { const int p2 = perm[i]; gi = p2 < n_old ? ei[p2] : idxs[p2 - n_old]; }
        }
        __syncthreads();
        if (tid < d) {
            mean[tid] = mu;
#pragma unroll
            for (int el = 0; el < ICF_MAX_NE; el++) if (el < ne) { eth[el * ldt + tid] = v[el]; xc[el * ldc + tid] = v[el] - mu; }
        } else if (tid >= 32 && tid - 32 < ne * NR) {
            eb[tid - 32] = gb;
            if (tid - 32 < ne) ei[tid - 32] = gi;
        }
        __syncthreads();
        // -- jnp.cov (ddof = 1) + 0.05 I, lower triangle, four columns per task  [compute_beta.py:61]
        if (cr >= 0) icf_cov_task(xc, C, ldc, ne, cr, cg);
        if (cr2 >= 0) icf_cov_task(xc, C, ldc, ne, cr2, cg2);
        __syncthreads();
        // latency build: this thread's d normals of the coming resampling are requested now and arrive while warp 0 factors
        float zpre[LAT ? d : 1];
        const bool pre = LAT && (S - ne) <= nt;
        if constexpr (LAT) {
            if (pre && tid < S - ne) {
                const float* zp = c.zb_iterT + (size_t)it * d * (S - ne) + tid;
#pragma unroll
                for (int k = 0; k < d; k++) zpre[k] = __ldg(zp + k * (S - ne));
            }
        }
        // -- Cholesky by warp 0, left-looking by panels of four columns, factor transposed in place (icf_chol_panel).  A two-warp look-ahead and a CTA-wide
        //    panel factorisation were measured here too and lost (DESIGN.md 5.4): under the 56-register cap the look-ahead spills, and with 12 chains per SM
        //    the phase is bound by issued instructions, not by warp 0's critical path.
        if constexpr (LAT) { if (warp == 0) icl_chol_regs<d>(C, lane); }       // latency build: register-resident right-looking factorisation (see icl_chol_regs)
        else if (warp == 0) icf_chol_panel<d>(C, ldc, lane);
        __syncthreads();
        // -- resample: one thread per new row, two columns per packed accumulator, k ascending  [compute_beta.py:63-66] (icf_mvn_row_unrolled).
        {
            constexpr int NG = (d + 3) / 4;
            const float* zT = c.zb_iterT + (size_t)it * d * nrow;
#pragma unroll 1
            for (int r = tid; r < nrow; r += nt) {
                pk::f2 acc[2 * NG];
                if constexpr (LAT) { if (pre) icf_mvn_row_regs<d>(LT, ldc, zpre, acc); else icf_mvn_row_unrolled<d>(LT, ldc, zT, nrow, r, acc); }
                else icf_mvn_row_unrolled<d>(LT, ldc, zT, nrow, r, acc);
                float* dst = th + r * ldt;
#pragma unroll
                for (int p = 0; p < NPAIR; p++) {
                    float x0, x1; pk::unpack(acc[p], x0, x1);
                    float v0 = mean[2 * p] + x0;
                    if (2 * p == nm) v0 = (v0 != v0) ? v0 : (v0 > c.sigma_clip ? v0 : c.sigma_clip);
                    dst[2 * p] = v0;
                    if (2 * p + 1 < d) {
                        float v1 = mean[2 * p + 1] + x1;
                        if (2 * p + 1 == nm) v1 = (v1 != v1) ? v1 : (v1 > c.sigma_clip ? v1 : c.sigma_clip);
                        dst[2 * p + 1] = v1;
                    }
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            resb[it] = ecost[0];
            if (it == c.iters_in - 1) {                // beta / reduced set of the best sample; sigma from the RESAMPLED array [Q7]
                for (int i = 0; i < NR; i++) { small[i] = eb[i]; ((int*)small)[16 + i] = (ei[0] >> (5 * i)) & 31; }
                const int p0 = perm[0];
                small[48] = p0 < ne ? eth[p0 * ldt + nm] : th[(p0 - ne) * ldt + nm];
            }
        }
        // the next iteration's first barrier (after the evaluation) orders these reads against later writes of perm / th
    }
    __syncthreads();
    // ---- hand the chosen reduced set to k_opt_risk (a separate kernel: the ~2000 SASS instructions of the risk evaluation would otherwise
    //      share the instruction cache with the 20-iteration loop of the other resident chains)
    if (tid < NR) { a.beta[(size_t)g * NR + tid] = small[tid]; ra.ridx[(size_t)g * NR + tid] = ((const int*)small)[16 + tid]; }
    if (tid == 0) a.sigma[g] = small[48];
}

// risk of the reduced set k_inner_cem_fast chose  [costs.py:173-186, 121-135]: thread (sample, r) re-rolls reduced rollout r from the
// sample's noisy controls (same arithmetic as the mother rollout => same bits) with the obstacle / lane maxima folded in, then one thread per
// sample evaluates the three MMD values.  The mother rollouts themselves are never stored.
#define OPT_RISK_THREADS 128
template <bool SORTED = false>
__global__ void __launch_bounds__(OPT_RISK_THREADS) k_opt_risk(DCfg c, RollArgs ra) {
    __shared__ float vals[3 * OPT_RISK_THREADS];
    const RiskArgs& a = ra.r;
    const int nr = c.nr, np = c.np, n = nr * np, tid = threadIdx.x;
    const int spb = OPT_RISK_THREADS / nr;
    const int ls = tid / nr, r = tid % nr, g = blockIdx.x * spb + ls;
    const bool live = ls < spb && g < a.n_samples;
    if (live) {
        const int e = g / a.B, mi = ra.ridx[(size_t)g * nr + r];
        const float* ct = ra.ctrl + (size_t)g * 2 * n;
        float m, l, u;
        if (ra.fold_risk) { const float* mr = ra.mrisk + ((size_t)g * nr * nr + mi) * 3; m = mr[0]; l = mr[1]; u = mr[2]; }     // folded by the mother rollout itself
        else rollout_risk<false, SORTED>(c, a, g, e, 0, ct + (mi / nr) * np, ct + n + (mi % nr) * np, a.state0 + e * 5,
                                 a.x_obs + (size_t)e * c.O * T_, a.y_obs + (size_t)e * c.O * T_, m, l, u);
        vals[tid] = m; vals[OPT_RISK_THREADS + tid] = l; vals[2 * OPT_RISK_THREADS + tid] = u;
    }
    __syncthreads();
    // the three MMD values of the sample [kernel_computation.py:67-87]: thread r evaluates kernel row r of each (ascending-j fma chains, 3 (nr + 1)
    // exponentials instead of 3 nr (nr + 1) on one thread), thread 0 of the sample folds the rows in ascending i -- the operations of mmd_cost in the same order
    __shared__ float rows_t[3 * OPT_RISK_THREADS], rows_u[3 * OPT_RISK_THREADS];
    if (live) {
        const float v = dm::kern_cost_v(c.kernel, a.sigma[g]);
        const int base = tid - r;
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const float* cst = vals + q * OPT_RISK_THREADS + base;
            const float ci = cst[r];
            float t = 0.0f;
            for (int j = 0; j < nr; j++) t = fmaf(dm::kern_cost(c.kernel, ci - cst[j], v), a.beta[(size_t)g * nr + j], t);
            const float e = dm::kern_cost(c.kernel, ci - 0.0f, v);
            float u = 0.0f;
            for (int j = 0; j < nr; j++) u = fmaf(e, c.beta_del, u);
            rows_t[q * OPT_RISK_THREADS + tid] = t; rows_u[q * OPT_RISK_THREADS + tid] = u;
        }
    }
    __syncthreads();
    if (live && r == 0) {
        float res[3];
#pragma unroll
        for (int q = 0; q < 3; q++) {
            float s1 = 0.0f, s2 = 0.0f;
            for (int i = 0; i < nr; i++) {
                const float bi = a.beta[(size_t)g * nr + i];
                s1 = fmaf(bi, rows_t[q * OPT_RISK_THREADS + tid + i], s1);
                s2 = fmaf(bi, rows_u[q * OPT_RISK_THREADS + tid + i], s2);
            }
            res[q] = c.ker_wt * (s1 - 2.0f * s2);
        }
        a.risk[g] = res[0];
        a.lane[g] = res[1] + res[2];
    }
}

// =====================================================================================================================================
// LATENCY build for launches of at most one chain per SM (batch = 1: 100 chains on 148 SMs; BASELINE's second headline, p50 per-solve latency).
// With an SM to itself a chain can spread each inner iteration over 16 warps instead of 3: the evaluation is split into (1) top-num_reduced per sample,
// (2) ONE kernel row sum per thread -- task (sample, reduced index): 25 of the 135 exponentials of a sample -- and (3) the per-sample KKT finish; the
// resampling runs one task per (row, group of four columns).  Same operations in the same order per element as k_inner_cem_fast (rows of a sample are
// independent IEEE chains there too), so the bits are unchanged; selection, gather, covariance and the one-warp panel Cholesky are shared code.
// Phase budget per inner iteration, batch 1 (DESIGN.md 5.1): 15 us -> ~9.5 us.
#define ICL_THREADS 512
// top-NR |theta| of a row (stable, ascending), packed 5 bits per index: first half of beta_sample_fast
template <int NR>
__device__ __forceinline__ int icl_topk(const float* __restrict__ row) {
    constexpr int nm = NR * NR;
    int tk[NR + 1];
#pragma unroll
    for (int p = 0; p <= NR; p++) tk[p] = 0;
    auto insert = [&](float x, int m) {
        const int v = (int)((dm::f2u(x) & 0x7fffffe0u) | (uint32_t)m);
        tk[0] = max(tk[0], v);
#pragma unroll
        for (int p = 0; p < NR; p++) { const int lo = min(tk[p], tk[p + 1]), hi = max(tk[p], tk[p + 1]); tk[p] = lo; tk[p + 1] = hi; }
    };
    if constexpr (NR == 5) {                       // the merge network of beta_sample_fast, unrolled (one chain per SM: code size is no concern here)
#define ICF_CE(a, b) { const int lo_ = min(a, b), hi_ = max(a, b); a = lo_; b = hi_; }
#pragma unroll
        for (int m = 0; m + 3 < nm; m += 4) {
            int s0 = (int)((dm::f2u(row[m]) & 0x7fffffe0u) | (uint32_t)m), s1 = (int)((dm::f2u(row[m + 1]) & 0x7fffffe0u) | (uint32_t)(m + 1));
            int s2 = (int)((dm::f2u(row[m + 2]) & 0x7fffffe0u) | (uint32_t)(m + 2)), s3 = (int)((dm::f2u(row[m + 3]) & 0x7fffffe0u) | (uint32_t)(m + 3));
            ICF_CE(s0, s1) ICF_CE(s2, s3) ICF_CE(s0, s2) ICF_CE(s1, s3) ICF_CE(s1, s2)
            tk[0] = max(tk[0], s3); tk[1] = max(tk[1], s2); tk[2] = max(tk[2], s1); tk[3] = max(tk[3], s0);
            ICF_CE(tk[0], tk[4]) ICF_CE(tk[1], tk[5]) ICF_CE(tk[0], tk[2]) ICF_CE(tk[1], tk[3]) ICF_CE(tk[0], tk[1]) ICF_CE(tk[2], tk[3]) ICF_CE(tk[4], tk[5])
        }
#undef ICF_CE
#pragma unroll
        for (int m = nm & ~3; m < nm; m++) insert(row[m], m);
    } else {
#pragma unroll
        for (int m = 0; m < nm; m++) insert(row[m], m);
    }
    int packed = 0; bool near = false;
#pragma unroll
    for (int p = 0; p < NR; p++) { packed |= (tk[p + 1] & 31) << (5 * p); near |= ((tk[p] ^ tk[p + 1]) < 32); }
    if (near) packed = top_abs_exact<NR>(row);
    return packed;
}
// sum_m k(D[row][m]; sigma), m ascending, two kernel entries per packed evaluation: one lane of beta_eval's row-sum loop
template <int NR, int KER>
__device__ __forceinline__ float icl_rowsum(const float* __restrict__ Drow, float sigma) {
    constexpr int nm = NR * NR;
    const LapK rinv2 = lap_k<false, KER>(sigma);
    float rs = 0.0f;
#pragma unroll 4
    for (int m = 0; m + 1 < nm; m += 2) {
        const pk::f2 e = lap2<false>(Drow[m], Drow[m + 1], rinv2);
        rs = rs + pk::lo(e); rs = rs + pk::hi(e);
    }
    if constexpr (nm & 1) rs = rs + pk::lo(lap2<false>(Drow[nm - 1], Drow[nm - 1], rinv2));
    return rs;
}
// reduced kernel, KKT solve and cost of one beta sample from its row sums: second half of beta_eval, operation for operation
template <int NR, int LDD, int KER>
__device__ __forceinline__ float icl_finish(const DCfg& c, int packed, float sigma, const float* __restrict__ rowsum, const float* __restrict__ D,
                                            float* __restrict__ beta_out) {
    constexpr int nm = NR * NR;
    const LapK rinv2 = lap_k<false, KER>(sigma);
    int ti[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) ti[i] = (packed >> (5 * i)) & 31;
    float K[NR][NR];
    {
        constexpr int NE = NR * (NR - 1) / 2;
        float dv[NE + 1];
        int e = 0;
#pragma unroll
        for (int i = 0; i < NR; i++) {
            K[i][i] = 1.0f;
#pragma unroll
            for (int j = 0; j < i; j++) dv[e++] = D[ti[i] * LDD + ti[j]];
        }
        dv[NE] = dv[NE - 1];
        float ev[NE + 1];
#pragma unroll
        for (int q = 0; q < NE; q += 2) pk::unpack(lap2<false>(dv[q], dv[q + 1], rinv2), ev[q], ev[q + 1]);
        e = 0;
#pragma unroll
        for (int i = 0; i < NR; i++)
#pragma unroll
            for (int j = 0; j < i; j++) { K[i][j] = ev[e]; K[j][i] = ev[e]; e++; }
    }
    float Lm[NR][NR], rd[NR];
#pragma unroll
    for (int j = 0; j < NR; j++) {
        float acc = K[j][j] + 0.05f;
#pragma unroll
        for (int k = 0; k < j; k++) acc = fmaf(-Lm[j][k], Lm[j][k], acc);
        float dd; dm::sqrt_rcp(acc, dd, rd[j]);
        Lm[j][j] = dd;
#pragma unroll
        for (int i = j + 1; i < NR; i++) {
            float aa = K[i][j];
#pragma unroll
            for (int k = 0; k < j; k++) aa = fmaf(-Lm[i][k], Lm[j][k], aa);
            Lm[i][j] = aa * rd[j];
        }
    }
    pk::f2 uw[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) {
        pk::f2 ab = pk::pack(c.inv_nm * rowsum[i], 1.0f);
#pragma unroll
        for (int k = 0; k < i; k++) ab = pk::fma2(pk::dup(-Lm[i][k]), uw[k], ab);
        uw[i] = pk::mul2(ab, pk::dup(rd[i]));
    }
#pragma unroll
    for (int i = NR - 1; i >= 0; i--) {
        pk::f2 ab = uw[i];
#pragma unroll
        for (int k = i + 1; k < NR; k++) ab = pk::fma2(pk::dup(-Lm[k][i]), uw[k], ab);
        uw[i] = pk::mul2(ab, pk::dup(rd[i]));
    }
    float u[NR], w[NR];
#pragma unroll
    for (int i = 0; i < NR; i++) pk::unpack(uw[i], u[i], w[i]);
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

// Latency kernel only: Cholesky of the d x d covariance by ONE warp with the whole lower triangle in registers (lane r holds row r), right-looking and fully
// unrolled: column j takes its pivot from lane j (one shuffle), every lane scales its entry, and the trailing entries (r, q), q > j, receive fma(-L_rj, L_qj, .)
// with L_qj shuffled from lane q.  Entry (r, q) therefore accumulates its k terms in ascending k and is then scaled by the pivot's reciprocal: the contract's order,
// the same bits as the panel versions.  No shared-memory round trip and no barrier inside the factorisation -- its critical path is pivot shuffle -> sqrt_rcp ->
// scale -> one fma per column (~2.4 k cycles for d = 26 against ~7 k for the two-warp look-ahead panels); 351 shuffles and ~1.2 k instructions of straight-line code,
// which only a kernel that has an SM to itself can afford.  The factor is written transposed with its zero fill (LT[k][q] = 0 for q < k) in one pass at the end.
template <int d>
__device__ __forceinline__ void icl_chol_regs(float* __restrict__ C, int lane) {
    constexpr int NG = (d + 3) / 4, ldc = (d + 3) & ~3;
    const int r = lane < d ? lane : d - 1;                 // lanes >= d shadow the last row (no stores)
    float a[4 * NG];
#pragma unroll
    for (int g = 0; g < NG; g++) {
        const float4 v = *reinterpret_cast<const float4*>(C + r * ldc + 4 * g);
        a[4 * g] = v.x; a[4 * g + 1] = v.y; a[4 * g + 2] = v.z; a[4 * g + 3] = v.w;
    }
    // Software pipeline: the NEXT column's pivot chain (shuffle -> sqrt -> reciprocal, ~85 cycles of pure latency) is started before the current column's trailing
    // updates (25 - j shuffles + fma, ~80 cycles of issue) and runs under them.  The next pivot is lane j+1's own diagonal entry, whose update needs no other lane
    // (L_qj of lane q IS its l): same operation, same bits as the generic update.  sqrt_rcp_fast is branch free, so chain and updates share one basic block; the
    // out-of-range case (uniform over the warp) is patched after the updates.
    float dd, rd;
    {
        const float a00 = __shfl_sync(FULL, a[0], 0);
        if (!dm::sqrt_rcp_fast(a00, dd, rd)) { const float2 v = dm::sqrt_rcp_slow(a00); dd = v.x; rd = v.y; }
    }
#pragma unroll
    for (int j = 0; j < d; j++) {
        const float l = lane == j ? dd : a[j] * rd;        // L[r][j] (meaningful for r >= j)
        a[j] = l;
        float ajn = 0.0f, ddn = 0.0f, rdn = 0.0f; bool okn = true;
        if (j + 1 < d) {
            ajn = __shfl_sync(FULL, fmaf(-l, l, a[j + 1]), j + 1);
            okn = dm::sqrt_rcp_fast(ajn, ddn, rdn);
        }
#pragma unroll
        for (int q = j + 1; q < d; q++) a[q] = fmaf(-l, __shfl_sync(FULL, l, q), a[q]);
        if (j + 1 < d) {
            if (!okn) { const float2 v = dm::sqrt_rcp_slow(ajn); ddn = v.x; rdn = v.y; }
            dd = ddn; rd = rdn;
        }
    }
    __syncwarp();
    if (lane < d) {
#pragma unroll
        for (int k = 0; k < d; k++) C[k * ldc + lane] = k <= lane ? a[k] : 0.0f;
    }
    __syncwarp();
}

template <int NR, int SC = 0, int NEC = 0, int KER = dm::KER_LAPLACE>          // SC / NEC: compile-time sample / elite counts, KER: kernel form, see k_inner_cem_fast
__global__ void __launch_bounds__(ICL_THREADS, 1) k_inner_cem_lat(DCfg c, RollArgs ra) {
    extern __shared__ __align__(128) float sm[];
    const RiskArgs& a = ra.r;
    const int g = blockIdx.x;
    if (g >= a.n_samples) return;
    constexpr int nm = NR * NR, d = nm + 1, NG = (d + 3) / 4, LDD = (nm + 3) & ~3;       // = FastLayout::ldd
    const int tid = threadIdx.x, nt = ICL_THREADS, warp = tid >> 5, lane = tid & 31;
    const int S = SC ? SC : c.S_in, ne = NEC ? NEC : c.n_el_in;
    const FastLayout L = fast_layout(NR, S, ne);
    const int ldt = L.ldt, ldc = L.ldc;
    float* D = sm + L.D; float* th = sm + L.th; float* cost = sm + L.cost; float* betas = ra.bscratch + (size_t)g * S * (NR + 1); int* idxs = (int*)(betas + S * NR);
    int* perm = (int*)(sm + L.perm); float* xc = sm + L.xc; float* C = sm + L.C; float* LT = C; float* mean = sm + L.mean;
    float* small = sm + L.small;
    float* eth = sm + L.eth;
    float* ecost = sm + L.ecost; float* eb = sm + L.ebetas; int* ei = (int*)(sm + L.eidxs);
    int* tis = (int*)(sm + L.total); float* rsum = sm + L.total + al4(S);        // per-sample reduced sets (packed) and row sums, behind the shared layout
    float* zs = rsum + al4(S * NR);                                              // this iteration's resampling normals [column][row], staged while warp 0 factors
    float* psum = zs + al4(d * (S - ne));                                        // look-ahead partial sums of the two-warp Cholesky, [2][32][4] (previous version; kept in the layout)
    {   // distance table of the mother features  [kernel_computation.py:31-33]; the features borrow the th region
        float* F = th;
        const float* Fg = ra.feat + (size_t)g * nm * 2 * NV;
#pragma unroll 1
        for (int i = tid; i < nm * 2 * NV; i += nt) F[i] = Fg[i];
        __syncthreads();
#pragma unroll 1
        for (int i = tid; i < nm * nm; i += nt) {
            const float* Fa = F + (i / nm) * 2 * NV; const float* Fb = F + (i % nm) * 2 * NV;
            float dist = 0.0f;
#pragma unroll 2
            for (int f = 0; f < 2 * NV; f++) dist = dm::kern_dist_acc<KER>(dist, Fa[f], Fb[f]);
            D[(i / nm) * LDD + i % nm] = dist;
        }
        __syncthreads();
    }
    int cr = -1, cg = 0;                                  // covariance task of this thread (d = 26: 98 tasks <= 512 threads)
    {
        int t = 0;
#pragma unroll 1
        for (int r = 0; r < d; r++) {
#pragma unroll 1
            for (int q4 = 0; q4 <= r / 4; q4++) { if (t == tid) { cr = r; cg = q4; } t++; }
        }
    }
    float* resb = a.res_beta + (size_t)g * c.iters_in;
#pragma unroll 1
    for (int it = 0; it < c.iters_in; it++) {
        const int n_old = it == 0 ? 0 : ne, n_new = S - n_old;
        const float* rows = it == 0 ? c.theta0 : th; const int rstride = it == 0 ? d : ldt;
        // -- evaluation in three phases
#pragma unroll 1
        for (int s = tid; s < n_new; s += nt) tis[s] = icl_topk<NR>(rows + s * rstride);
        __syncthreads();
#pragma unroll 1
        for (int task = tid; task < n_new * NR; task += nt) {
            const int s = task / NR, i = task - s * NR;
            rsum[task] = icl_rowsum<NR, KER>(D + ((tis[s] >> (5 * i)) & 31) * LDD, rows[s * rstride + nm]);
        }
        __syncthreads();
#pragma unroll 1
        for (int s = tid; s < n_new; s += nt) {
            cost[s] = icl_finish<NR, LDD, KER>(c, tis[s], rows[s * rstride + nm], rsum + s * NR, D, betas + s * NR);
            idxs[s] = tis[s];
        }
        __syncthreads();
        if (warp == 0) icf_select(lane, S, n_old, ne, ecost, cost, perm, ecost);      // (a CTA-wide rank count, 4 threads per candidate, was measured here: its two extra block barriers cost more than the one-warp rounds, 4.79 vs 4.71 ms)
        __syncthreads();
        float v[ICF_MAX_NE]; float mu = 0.0f, gb = 0.0f; int gi = 0;
        if (tid < d) {
            float s = 0.0f;
#pragma unroll
            for (int el = 0; el < ICF_MAX_NE; el++) {
                if (el < ne) {
                    const int p = perm[el];
                    v[el] = p < n_old ? eth[p * ldt + tid] : rows[(p - n_old) * rstride + tid];
                    s = s + v[el];
                }
            }
            mu = s / (float)ne;
        } else if (tid >= 32 && tid - 32 < ne * NR) {
            const int i = tid - 32, p = perm[i / NR], k = i % NR;
            gb = p < n_old ? eb[p * NR + k] : betas[(p - n_old) * NR + k];
            if (i < ne) { const int p2 = perm[i]; gi = p2 < n_old ? ei[p2] : idxs[p2 - n_old]; }
        }
        __syncthreads();
        if (tid < d) {
            mean[tid] = mu;
#pragma unroll
            for (int el = 0; el < ICF_MAX_NE; el++) if (el < ne) { eth[el * ldt + tid] = v[el]; xc[el * ldc + tid] = v[el] - mu; }
        } else if (tid >= 32 && tid - 32 < ne * NR) {
            eb[tid - 32] = gb;
            if (tid - 32 < ne) ei[tid - 32] = gi;
        }
        __syncthreads();
        if (cr >= 0) icf_cov_task(xc, C, ldc, ne, cr, cg);
        __syncthreads();
        if (warp == 0) icl_chol_regs<d>(C, lane);          // (a two-warp look-ahead panel factorisation was the previous version: 3.7 us per factorisation against ~1.7)
        else if (warp >= 2) {                             // the other warps fetch the iteration's normals (first touch: L2 latency) behind the Cholesky
            // eight independent loads in flight per thread, then the stores: rolled one at a time, each thread paid the L2 / DRAM latency of a first touch six times in
            // a row (the ncu source page showed this phase waiting on these stores, not on the factorisation)
            const float* zg = c.zb_iterT + (size_t)it * d * (S - ne);
            const int nz = d * (S - ne), st = nt - 64;
#pragma unroll 1
            for (int i0 = tid - 64; i0 < nz; i0 += 8 * st) {
                float t8[8];
#pragma unroll
                for (int u = 0; u < 8; u++) t8[u] = i0 + u * st < nz ? __ldg(zg + i0 + u * st) : 0.0f;
#pragma unroll
                for (int u = 0; u < 8; u++) if (i0 + u * st < nz) zs[i0 + u * st] = t8[u];
            }
        }
        __syncthreads();
        {   // resample: task = (new row r, group of four columns g4); columns 4 g4 .. 4 g4 + 3 take k = 0 .. 4 g4 + 3 ascending (icf_mvn_row_unrolled's order)
            const int nrow = S - ne;
            const float* zT = zs;
#pragma unroll 1
            for (int task = tid; task < nrow * NG; task += nt) {
                // column group g4 costs 4 g4 + 4 steps: the longest groups go to the first pass, so the (partial) second pass holds the shortest tasks
                const int gq = task / nrow, g4 = NG - 1 - gq, r = task - gq * nrow;
                const int kend = min(4 * g4 + 3, d - 1);
                pk::f2 a01 = pk::dup(0.0f), a23 = pk::dup(0.0f);
#pragma unroll 4
                for (int k = 0; k <= kend; k++) {
                    const pk::f2 z2 = pk::dup(zT[k * nrow + r]);
                    const float4 l = *reinterpret_cast<const float4*>(LT + k * ldc + 4 * g4);
                    a01 = pk::fma2(pk::pack(l.x, l.y), z2, a01); a23 = pk::fma2(pk::pack(l.z, l.w), z2, a23);
                }
                float x[4]; pk::unpack(a01, x[0], x[1]); pk::unpack(a23, x[2], x[3]);
                float* dst = th + r * ldt + 4 * g4;
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int q = 4 * g4 + u;
                    if (q < d) {
                        float vv = mean[q] + x[u];
                        if (q == nm) vv = (vv != vv) ? vv : (vv > c.sigma_clip ? vv : c.sigma_clip);
                        dst[u] = vv;
                    }
                }
            }
        }
        __syncthreads();
        if (tid == 0) {
            resb[it] = ecost[0];
            if (it == c.iters_in - 1) {
                for (int i = 0; i < NR; i++) { small[i] = eb[i]; ((int*)small)[16 + i] = (ei[0] >> (5 * i)) & 31; }
                const int p0 = perm[0];
                small[48] = p0 < ne ? eth[p0 * ldt + nm] : th[(p0 - ne) * ldt + nm];
            }
        }
    }
    __syncthreads();
    if (tid < NR) { a.beta[(size_t)g * NR + tid] = small[tid]; ra.ridx[(size_t)g * NR + tid] = ((const int*)small)[16 + tid]; }
    if (tid == 0) a.sigma[g] = small[48];
}
