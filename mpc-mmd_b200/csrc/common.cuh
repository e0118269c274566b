// common.cuh -- device-side configuration / workspace structs and small contract helpers shared
// by the kernels of libmpcmmd.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "dmath.cuh"
#include "drng.cuh"

#define T_ 100      // num   (reference S/optimizer/cem.py:38)
#define NV 11       // nvar  (cem.py:50)
#define NL 99       // lane rows per side (cem.py:126-134)
#define NPAR 8      // num_params (cem.py:136)
#define FULL 0xffffffffu
#define MPCMMD_MAX_NR_DEV 64   // local-array bound for num_reduced in the num_reduced-rollout risk paths (cvar / saa / mmd_random)

struct DCfg {
    int B, np, nr, nm, O, iters, n_el, n_el_cost, noise_kind, S_in, iters_in, n_el_in;
    float sigma_acc, sigma_steer, ksig_steer, acc_const, steer_const, beta_a, beta_b;
    float v_min, v_max, a_max, b_lane_ub, b_lane_lb, y_lb, y_ub, a2_obs, b2_obs;
    float wheel_base, dt, steer_max, steer_rate_pen, alpha_quant, ker_wt;
    float lam_inv, one_m_alpha_mean, alpha_mean, one_m_alpha_cov, alpha_cov;
    float sigma_clip, inv_nm, m2_inv_nm, beta_del, sigma_random;
    float obs_win;                                           // half-width of the x window outside of which the obstacle indicator is exactly 0: sqrt(a2_obs) + 0.01
    int kernel;                                              // MMD kernel form (dm::KER_*) of the scalar-cost MMD (the inner-CEM kernels take it as a template argument); fills the
                                                             // alignment gap before the pointers, so no other member moves
    const float *P, *Pd, *Pdd, *Gx, *Gy, *Kx, *Ky, *Wfit;   // device copies of the host constants
    const float* proj_const;                                 // P | Pd | Pdd | Gx | Gy | Kx | Ky as ONE 16-byte-aligned block (bulk-copied into shared memory by k_project)
    const float* proj_tc_const;                              // tf32 (hi, lo) images of P / Pd / Pdd + Gx | Gy | Kx | Ky for k_project_tc
    const float *z_init, *theta0, *zb_iter;                  // constant normal tables (generated at create)
    const float *theta0T;                                    // theta0 transposed to [column][row]
    const float *zb_iterT;                                   // zb_iter transposed to [iter][column][row] for coalesced row-per-thread reads
};

// per-batch device workspace; every array is [episode][...] with the strides noted
struct DWork {
    float *params;                 // [E][B][8]
    float *lam_x, *lam_y;          // [E][B][11]
    float *s_lane;                 // [E][B][198]
    float *mean, *cov;             // [E][8], [E][64]
    float *cx, *cy;                // [E][B][11]
    float *res_norm, *cost_base;   // [E][B]
    float *acc, *steer;            // [E][B][100]
    float *risk, *lane;            // [E][B]
    float *beta, *sigma, *res_beta;// [E][B][nr], [E][B], [E][B][iters_in]
    float *z1, *z2, *z3;           // [E][iters][nr*np]
    float *zcem;                   // [E][iters][(B-n_el)*8]
    uint32_t *keys;                // [E][iters][4]
    float *btab;                   // [E][iters][4][GT_FIELDS][nr*np]  Beta-sampler candidate table (beta noise only)
    // staged inputs
    int32_t *idx_mpc;              // [E]
    float *init_state;             // [E][6]
    float *mean0, *cov0;           // [E][8], [E][64]
    float *x_obs, *y_obs;          // [E][O][100]
    float *sx_obs, *sy_obs;        // [E][100][O]  obstacle positions per knot, sorted by x (k_obs_sort; only for num_obs > OBS_SORT_MIN, else null)
    int *obs_nan;                  // [E][100]     1 if a coordinate of that knot is NaN (then the plain loop runs)
    float *v_des;                  // [E]
    // staged outputs
    float *o_cx, *o_cy, *o_lane, *o_obs, *o_beta, *o_sigma, *o_res_beta;
    int32_t *o_sel;                // [E][iters]
};

// ---- TMA bulk copy global -> shared with mbarrier completion (cp.async.bulk, sm_90+): one elected thread issues the copy, every thread of
// the CTA waits on the barrier's phase.  `bytes` must be a multiple of 16, both addresses 16-byte aligned.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, unsigned long long* bar) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long* bar, uint32_t parity) {
    asm volatile("{\n\t.reg .pred p;\n\tWAIT_%=:\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t@p bra DONE_%=;\n\tbra WAIT_%=;\n\tDONE_%=:\n\t}"
                 :: "r"(smem_u32(bar)), "r"(parity) : "memory");
}

// xor-butterfly sum over the 32 lanes (every lane ends with the same value; matches the oracle's
// lane_sum_sq combine order 16,8,4,2,1)
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v = v + __shfl_xor_sync(FULL, v, off);
    return v;
}
// NaN-propagating max over the warp (order-independent)
__device__ __forceinline__ float warp_nmax(float v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) v = dm::nmax_(v, __shfl_xor_sync(FULL, v, off));
    return v;
}
__device__ __forceinline__ float dot11(const float* row, const float* c) {
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < NV; k++) acc = fmaf(row[k], c[k], acc);
    return acc;
}
// Cholesky of a tiny row-major matrix by ONE thread (8x8 CEM covariance); same op order as the contract
__device__ __forceinline__ void chol_serial(float* A, int n, int ld, float* rd) {
    for (int j = 0; j < n; j++) {
        float acc = A[j * ld + j];
        for (int k = 0; k < j; k++) acc = fmaf(-A[j * ld + k], A[j * ld + k], acc);
        float d = sqrtf(acc);
        A[j * ld + j] = d;
        rd[j] = 1.0f / d;
        for (int i = j + 1; i < n; i++) {
            float a = A[i * ld + j];
            for (int k = 0; k < j; k++) a = fmaf(-A[i * ld + k], A[j * ld + k], a);
            A[i * ld + j] = a * rd[j];
        }
    }
}
__device__ __forceinline__ float mvn_elem(const float* L, int ld, int i, const float* z, float mean) {
    float acc = 0.0f;
    for (int k = 0; k <= i; k++) acc = fmaf(L[i * ld + k], z[k], acc);
    return mean + acc;
}
