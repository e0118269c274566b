// mpcmmd_api.cu -- C ABI of libmpcmmd.so (see include/mpcmmd.h): handle lifetime, the batched
// solve (one CUDA graph of 3 + (3 or 4)*maxiter_cem kernels per (cost kind, episode count)) and the
// stage entry points used by the teacher-forced parity tests.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <math.h>
#include <string.h>
#include <map>
#include <mutex>
#include <string>
#include <vector>
#include "../../include/mpcmmd.h"
#include "k_project.cuh"
#include "k_project_tc.cuh"
#include "k_risk.cuh"
#include "k_inner_cem.cuh"
#include "k_inner_cem_warp.cuh"
#include "k_inner_split.cuh"
#include "k_inner_pipe.cuh"
#include "k_inner_big.cuh"
#include "k_select.cuh"
#include "k_validate.cuh"
#include "k_validate_noise.cuh"
#include "k_validate_jax.cuh"

static thread_local std::string g_err;
static int fail(const std::string& m) { g_err = m; return -1; }
#define CK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return fail(std::string(#x) + ": " + cudaGetErrorString(e_)); } while (0)

extern "C" const char* mpcmmd_last_error(void) { return g_err.c_str(); }

// Dynamic shared memory opt-in of a kernel is a per-(device, function) attribute shared by every handle of the process: it is only ever RAISED
// (a second handle with a smaller configuration must not lower the limit under a live handle whose graphs ask for more).
static std::mutex g_smem_mu;
static std::map<std::pair<int, const void*>, size_t> g_smem_max;
static int raise_smem(int device, const void* fn, size_t bytes, bool carveout_max = false) {
    std::lock_guard<std::mutex> lk(g_smem_mu);
    size_t& cur = g_smem_max[std::make_pair(device, fn)];
    if (bytes > cur) {
        if (bytes > 48 * 1024 || cur > 0) CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
        cur = bytes;
    }
    if (carveout_max) CK(cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    return 0;
}
extern "C" int mpcmmd_version(void) { return 100; }

#define MAX_GROUPS 8
struct mpcmmd_handle_s {
    int device = 0;
    mpcmmd_config cfg;         // host copy (matrix pointers are NOT valid after create)
    DCfg d;
    DWork w;
    float *beq_x = nullptr, *beq_y = nullptr, *state0 = nullptr;   // [E][3], [E][4], [E][5]
    float *xroll = nullptr, *yroll = nullptr, *feat = nullptr;     // mmd_opt scratch (ensure_opt_scratch)
    float *rolls_x = nullptr, *rolls_y = nullptr;                  // [E*B][nm][np] mother rollouts (generic / warp-per-chain inner kernels only)
    int* ridx = nullptr;       // [E*B][nr] reduced sets (k_inner_cem_fast -> k_opt_risk)
    float* bscratch = nullptr; // [E*B][S][nr+1] row records of k_inner_cem_fast
    float* ctrl = nullptr;     // [E*B][2][nr*np] noisy controls (k_rollouts -> k_opt_risk)
    float* mrisk = nullptr;         // [E*B][nm][3] obstacle / lane maxima of the mother rollouts (small mmd_opt launches: RollArgs::fold_risk)
    float* throws = nullptr;        // [E*B][nm+1][ICP_TH_LD] candidate-elite rows of the pipelined inner CEM (k_inner_pipe.cuh)
    int pipe_minb = 8;              // CTAs per SM the pipelined kernel is compiled for (MPCMMD_PIPE_MINB=8|9|12)
    float* big_state = nullptr;     // [big_chunk][BigLayout::total] chain blocks of k_inner_cem_big (num_reduced > 10), reused by successive chain ranges
    int big_chunk = 0;
    float* split_state = nullptr;   // [E*B][SplitLayout::total] chain blocks of the phase-split inner CEM (k_inner_split.cuh)
    float* stash = nullptr;    // row stash of k_inner_cem_warp, [warp_grid][S][32]
    int warp_grid = 0;         // persistent CTAs of k_inner_cem_warp (SMs x resident CTAs per SM)
    int sm_count = 148;
    int inner_mode = 0;        // 0 auto, 1 warp-per-chain, 2 CTA-per-chain, 3 generic, 4 CTA-per-chain latency build, 5 phase-split (MPCMMD_INNER_CEM=auto|warp|cta|generic|lat|split)
    int E = 0;
    bool fast_math = false;    // MPCMMD_MATH=fast: Laplace-kernel exponentials of the inner CEM on MUFU.EX2 (opt-in, tolerance parity only)
    bool proj_tc = false;      // MPCMMD_PROJ=tc: tensor-core projection kernel (k_project_tc)
    bool proj_tc_always = false;
    std::vector<void*> allocs;
    std::map<std::pair<int, int>, cudaGraphExec_t> graphs;
    std::map<std::pair<int, int>, int> graph_launches;
    int last_launches = 0;
    cudaStream_t own_stream = nullptr;
    cudaStream_t aux_stream[MAX_GROUPS - 1] = {};   // further branches of a solve graph whose episodes are split into groups (see solve_groups)
    cudaEvent_t ev_fork = nullptr, ev_join[MAX_GROUPS - 1] = {};
    int groups_override = 0;                 // MPCMMD_GROUPS=1..8: force the number of episode groups of a solve graph (0 = automatic)
    int prio_mode = 0;                       // MPCMMD_PRIO=0|1|2 (experiment, default off): highest stream priority on the kernel nodes of mmd_opt graphs (1) / of the other cost functions' graphs (2)
};

// ---- episode-offset view of a handle's workspace: every per-episode array advanced by e0 episodes.  A solve graph can then enqueue disjoint episode
// ranges on different streams with the unchanged launch code (episodes are independent; sample index g and episode index e stay relative to the view).
struct ViewSave { DWork w; float *beq_x, *beq_y, *state0, *feat, *ctrl, *bscratch, *throws, *split_state, *rolls_x, *rolls_y, *xroll, *mrisk; int* ridx; };
static ViewSave push_view(mpcmmd_handle_s* h, int e0) {
    ViewSave sv = {h->w, h->beq_x, h->beq_y, h->state0, h->feat, h->ctrl, h->bscratch, h->throws, h->split_state, h->rolls_x, h->rolls_y, h->xroll, h->mrisk, h->ridx};
    if (e0 == 0) return sv;
    const DCfg& d = h->d; DWork& w = h->w;
    const size_t e = (size_t)e0, B = d.B, n = (size_t)d.nr * d.np, ncem = (size_t)(d.B - d.n_el) * NPAR, it = d.iters;
#define ADV(p, stride) if (p) p += e * (stride)
    ADV(w.params, B * NPAR); ADV(w.lam_x, B * NV); ADV(w.lam_y, B * NV); ADV(w.s_lane, B * 2 * NL); ADV(w.mean, NPAR); ADV(w.cov, 64);
    ADV(w.cx, B * NV); ADV(w.cy, B * NV); ADV(w.res_norm, B); ADV(w.cost_base, B); ADV(w.acc, B * T_); ADV(w.steer, B * T_); ADV(w.risk, B); ADV(w.lane, B);
    ADV(w.beta, B * d.nr); ADV(w.sigma, B); ADV(w.res_beta, B * d.iters_in); ADV(w.z1, it * n); ADV(w.z2, it * n); ADV(w.z3, it * n); ADV(w.zcem, it * ncem);
    ADV(w.keys, it * 4); ADV(w.btab, it * 4 * GT_FIELDS * n); ADV(w.idx_mpc, 1); ADV(w.init_state, 6); ADV(w.mean0, NPAR); ADV(w.cov0, 64);
    ADV(w.x_obs, (size_t)d.O * T_); ADV(w.y_obs, (size_t)d.O * T_); ADV(w.v_des, 1);
    ADV(w.sx_obs, (size_t)d.O * T_); ADV(w.sy_obs, (size_t)d.O * T_); ADV(w.obs_nan, T_);
    ADV(w.o_cx, NV); ADV(w.o_cy, NV); ADV(w.o_lane, 1); ADV(w.o_obs, 1); ADV(w.o_beta, d.nr); ADV(w.o_sigma, 1); ADV(w.o_res_beta, d.iters_in); ADV(w.o_sel, it);
    ADV(h->beq_x, 3); ADV(h->beq_y, 4); ADV(h->state0, 5);
    ADV(h->feat, B * d.nm * 2 * NV); ADV(h->ctrl, B * 2 * n); ADV(h->ridx, B * d.nr); ADV(h->bscratch, B * d.S_in * (d.nr + 1));
    ADV(h->throws, B * (d.nm + 1) * ICP_TH_LD); ADV(h->split_state, B * (size_t)split_layout(d.nr, d.S_in, d.n_el_in).total);
    ADV(h->rolls_x, B * d.nm * d.np); ADV(h->rolls_y, B * d.nm * d.np); ADV(h->mrisk, B * d.nm * 3);
    if (h->xroll) h->xroll = h->feat;
#undef ADV
    return sv;
}
static void pop_view(mpcmmd_handle_s* h, const ViewSave& sv) {
    h->w = sv.w; h->beq_x = sv.beq_x; h->beq_y = sv.beq_y; h->state0 = sv.state0; h->feat = sv.feat; h->ctrl = sv.ctrl; h->bscratch = sv.bscratch;
    h->throws = sv.throws; h->split_state = sv.split_state; h->rolls_x = sv.rolls_x; h->rolls_y = sv.rolls_y; h->xroll = sv.xroll; h->mrisk = sv.mrisk; h->ridx = sv.ridx;
}

template <typename Tp>
static int dalloc(mpcmmd_handle_s* h, Tp** p, size_t n) {
    void* q = nullptr;
    CK(cudaMalloc(&q, (n ? n : 1) * sizeof(Tp)));
    CK(cudaMemset(q, 0, (n ? n : 1) * sizeof(Tp)));
    h->allocs.push_back(q);
    *p = (Tp*)q;
    return 0;
}
static int upload(mpcmmd_handle_s* h, const float** dst, const float* src, size_t n) {
    if (!src) return fail("mpcmmd_create: null matrix pointer in config");
    float* q = nullptr;
    if (dalloc(h, &q, n)) return -1;
    CK(cudaMemcpy(q, src, n * sizeof(float), cudaMemcpyHostToDevice));
    *dst = q;
    return 0;
}

// k_init also prepares the per-episode boundary vectors (cem_helper.py:152-167, cem.py:218-219)
__global__ void k_boundary(const float* init_state, float* beq_x, float* beq_y, float* state0, int n_ep) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_ep) return;
    const float* s = init_state + e * 6;    // x, y, vx, vy, ax, ay
    beq_x[e * 3 + 0] = s[0]; beq_x[e * 3 + 1] = s[2]; beq_x[e * 3 + 2] = s[4];
    beq_y[e * 4 + 0] = s[1]; beq_y[e * 4 + 1] = s[3]; beq_y[e * 4 + 2] = s[5]; beq_y[e * 4 + 3] = 0.0f;
    state0[e * 5 + 0] = s[0]; state0[e * 5 + 1] = s[1]; state0[e * 5 + 2] = s[2]; state0[e * 5 + 3] = s[3];
    state0[e * 5 + 4] = dm::atan2_(s[3], s[2]);
}

// the packed-FP32 kernel (k_inner_cem.cuh) covers num_reduced^2 + 1 <= 32 with at most 128 candidates / 12 elites per inner iteration;
// everything else runs the generic kernel of k_risk.cuh
static bool inner_cem_is_fast(const DCfg& d) {
    return d.nr <= 5 && d.S_in <= ICF_MAX_S && d.n_el_in <= ICF_MAX_NE && d.n_el_in >= 2 && d.S_in - d.n_el_in >= 1;
}
// samples per CTA of k_rollouts: as many as keep one thread per rollout busy (bounded by shared memory), but never so
// many that a small batch leaves SMs idle (latency at batch = 1 episode)
// latency regime of the num_reduced-rollout costs: with one thread per rollout the launch cannot fill the GPU, so the controls are drawn by
// whole CTAs first (RollArgs::stage_ctrl)
static int roll_stage_ctrl(const mpcmmd_handle_s* h, int kind, int n_samples) {
    return kind != MPCMMD_COST_MMD_OPT && (long long)n_samples * h->d.nr < 2LL * h->sm_count * ROLL_THREADS;
}
static int roll_spb(const mpcmmd_handle_s* h, int kind, int n_samples) {
    const DCfg& d = h->d;
    const int R = (kind == MPCMMD_COST_MMD_OPT) ? d.nm : d.nr;
    const int stage = roll_stage_ctrl(h, kind, n_samples);
    int spb = ROLL_THREADS / R; if (spb < 1) spb = 1; if ((kind == MPCMMD_COST_MMD_OPT || stage) && spb > 8) spb = 8;
    while (spb > 1 && (size_t)roll_smem_floats(spb, d.nr, d.np, R, stage) * sizeof(float) > 96 * 1024) spb--;
    while (spb > 1 && (n_samples + spb - 1) / spb < 4 * h->sm_count) spb--;
    // latency regime of the num_reduced-rollout costs: the control draws of a sample are spread over the whole CTA, so few samples per CTA shorten the serial
    // staging (measured at 25 / 50 episodes: cvar 3.34 / 5.88 ms with up to 4 samples per CTA, 2.89 / 4.74 ms with 2)
    if (stage && spb > 2) spb = 2;
    return spb;
}
static size_t roll_smem_for(const DCfg& d, int kind, int spb, int stage, int fold = 0) {
    const int R = (kind == MPCMMD_COST_MMD_OPT) ? d.nm : d.nr;
    return (size_t)roll_smem_floats(spb, d.nr, d.np, R, stage, fold) * sizeof(float);
}
// largest dynamic shared memory any launch of this handle can ask for (opt-in at create)
static size_t roll_smem(const mpcmmd_handle_s* h, int kind) {
    const DCfg& d = h->d;
    const size_t a = roll_smem_for(d, kind, roll_spb(h, kind, 1 << 30), 0), b = roll_smem_for(d, kind, roll_spb(h, kind, 1), roll_stage_ctrl(h, kind, 1));
    size_t c = 0;
    for (int spb = 1; spb <= 8; spb++) { const size_t v = roll_smem_for(d, kind, spb, kind != MPCMMD_COST_MMD_OPT); if (v <= 96 * 1024 && v > c) c = v; }
    if (kind == MPCMMD_COST_MMD_OPT && inner_cem_is_fast(d)) { const size_t v = roll_smem_for(d, kind, 1, 0, 1); if (v > c) c = v; }      // latency regime (num_reduced <= 5 only): positions of one sample's mother rollouts
    return a > b ? (a > c ? a : c) : (b > c ? b : c);
}
// k_rollouts instantiation of a launch: mode (ROLL_*), noise path (NZ_*), sorted obstacle windows (ROLL_FLY only; Gaussian or the run-time noise path)
static const void* rollouts_kernel(int mode, int nz, int sorted, int ov = OV_PLAIN) {
#define RK_NZ(M, S, O) (nz == NZ_GAUSS ? (const void*)k_rollouts<M, S, NZ_GAUSS, O> : nz == NZ_BETA_TABLE ? (const void*)k_rollouts<M, S, NZ_BETA_TABLE, O> : (const void*)k_rollouts<M, S, NZ_ANY, O>)
    if (mode == ROLL_OPT) return ov == OV_FOLD ? RK_NZ(ROLL_OPT, false, OV_FOLD) : ov == OV_WRITE ? RK_NZ(ROLL_OPT, false, OV_WRITE) : RK_NZ(ROLL_OPT, false, OV_PLAIN);
    if (mode == ROLL_STAGED) return RK_NZ(ROLL_STAGED, false, OV_PLAIN);
    if (sorted) return nz == NZ_GAUSS ? (const void*)k_rollouts<ROLL_FLY, true, NZ_GAUSS> : (const void*)k_rollouts<ROLL_FLY, true, NZ_ANY>;
    return RK_NZ(ROLL_FLY, false, OV_PLAIN);
#undef RK_NZ
}
typedef void (*inner_cem_fn)(DCfg, RollArgs);
enum { INNER_WARP = 1, INNER_CTA = 2, INNER_GENERIC = 3, INNER_CTA_LAT = 4, INNER_SPLIT = 5, INNER_PIPE = 6, INNER_CTA_FASTMATH = 7, INNER_BIG = 8, INNER_LAT512 = 9 };
#define MPCMMD_BIG_SCRATCH_BYTES ((size_t)8 << 30)      // global chain state of k_inner_cem_big held at a time (num_reduced 40: 23 MB per chain)
#define INNER_DEFAULT_THROUGHPUT INNER_CTA
typedef void (*pipe_fn)(DCfg, RollArgs, float*);
// the pipelined kernel stages the mother features through its row buffer: (S - ne) rows of nm + 1 (odd stride) must hold nm x 22 floats
static bool pipe_ok(const DCfg& d) { return inner_cem_is_fast(d) && (d.S_in - d.n_el_in) * ((d.nm + 1) | 1) >= d.nm * 2 * NV; }
static pipe_fn pipe_kernel(int nr, int minb) {
#define PK(N) (minb >= 12 ? k_inner_cem_pipe<N, 12> : minb == 9 ? k_inner_cem_pipe<N, 9> : k_inner_cem_pipe<N, 8>)
    switch (nr) { case 2: return PK(2); case 3: return PK(3); case 4: return PK(4); case 5: return PK(5); default: return nullptr; }
#undef PK
}
typedef void (*split_dist_fn)(DCfg, SplitArgs);
typedef void (*split_it_fn)(DCfg, SplitArgs, int);
struct SplitKernels { split_dist_fn dist; split_it_fn eval, update; };
static SplitKernels split_kernels(int nr) {
    switch (nr) {
        case 2: return {k_icem_dist<2>, k_icem_eval<2>, k_icem_update<2>};
        case 3: return {k_icem_dist<3>, k_icem_eval<3>, k_icem_update<3>};
        case 4: return {k_icem_dist<4>, k_icem_eval<4>, k_icem_update<4>};
        case 5: return {k_icem_dist<5>, k_icem_eval<5>, k_icem_update<5>};
        default: return {nullptr, nullptr, nullptr};
    }
}
static size_t split_eval_smem(const DCfg& d) { const int dd = d.nm + 1; return (size_t)(al4(d.nm * d.nm) + (dd + 1) * al4(dd)) * sizeof(float); }
static size_t split_update_smem(const DCfg& d) { return (size_t)ICU_WARPS * upd_layout(d.nr).total * sizeof(float); }
static int g_chol = 0;       // MPCMMD_CHOL=panel|la|cta (read at create): Cholesky build of the specialised throughput kernel (0 one-warp panels, 1 two-warp look-ahead, 2 CTA-wide panels)
// KER = MMD kernel form (dm::KER_*).  The experimental warp-per-chain kernel and the Cholesky variants exist for Laplace only (a Gaussian handle refuses them at create)
template <int KER>
static inner_cem_fn inner_cem_kernel_k(const DCfg& d, int kind) {
    if constexpr (KER == dm::KER_LAPLACE) {
        if (kind == INNER_WARP) switch (d.nr) {
            case 2: return k_inner_cem_warp<2>; case 3: return k_inner_cem_warp<3>; case 4: return k_inner_cem_warp<4>; case 5: return k_inner_cem_warp<5>;
        }
        if (d.nr == 5 && d.S_in == 100 && d.n_el_in == 11) {
            if (kind == INNER_CTA && g_chol == 1) return k_inner_cem_fast<5, false, false, 100, 11, 1>;
            if (kind == INNER_CTA && g_chol == 2) return k_inner_cem_fast<5, false, false, 100, 11, 2>;
        }
    } else if (kind == INNER_WARP) return nullptr;
    if (d.nr == 5 && d.S_in == 100 && d.n_el_in == 11) {          // the reference's sizes as compile-time constants
        if (kind == INNER_CTA) return k_inner_cem_fast<5, false, false, 100, 11, 0, KER>;
        if (kind == INNER_CTA_LAT) return k_inner_cem_fast<5, true, false, 100, 11, 0, KER>;
        if (kind == INNER_CTA_FASTMATH) return k_inner_cem_fast<5, false, true, 100, 11, 0, KER>;
        if (kind == INNER_LAT512) return k_inner_cem_lat<5, 100, 11, KER>;
    }
    if (kind == INNER_CTA) switch (d.nr) {
        case 2: return k_inner_cem_fast<2, false, false, 0, 0, 0, KER>; case 3: return k_inner_cem_fast<3, false, false, 0, 0, 0, KER>;
        case 4: return k_inner_cem_fast<4, false, false, 0, 0, 0, KER>; case 5: return k_inner_cem_fast<5, false, false, 0, 0, 0, KER>;
    }
    if (kind == INNER_LAT512) switch (d.nr) {
        case 2: return k_inner_cem_lat<2, 0, 0, KER>; case 3: return k_inner_cem_lat<3, 0, 0, KER>; case 4: return k_inner_cem_lat<4, 0, 0, KER>; case 5: return k_inner_cem_lat<5, 0, 0, KER>;
    }
    if (kind == INNER_CTA_FASTMATH) switch (d.nr) {
        case 2: return k_inner_cem_fast<2, false, true, 0, 0, 0, KER>; case 3: return k_inner_cem_fast<3, false, true, 0, 0, 0, KER>;
        case 4: return k_inner_cem_fast<4, false, true, 0, 0, 0, KER>; case 5: return k_inner_cem_fast<5, false, true, 0, 0, 0, KER>;
    }
    if (kind == INNER_CTA_LAT) switch (d.nr) {
        case 2: return k_inner_cem_fast<2, true, false, 0, 0, 0, KER>; case 3: return k_inner_cem_fast<3, true, false, 0, 0, 0, KER>;
        case 4: return k_inner_cem_fast<4, true, false, 0, 0, 0, KER>; case 5: return k_inner_cem_fast<5, true, false, 0, 0, 0, KER>;
    }
    if (d.S_in == 100 && d.n_el_in == 11) switch (d.nr) {       // the reference's sizes as compile-time constants (generic kernel, num_reduced 6..10)
        case 6: return k_inner_cem<6, 100, 11, KER>; case 7: return k_inner_cem<7, 100, 11, KER>; case 8: return k_inner_cem<8, 100, 11, KER>;
        case 9: return k_inner_cem<9, 100, 11, KER>; case 10: return k_inner_cem<10, 100, 11, KER>;
    }
    switch (d.nr) {
        case 2: return k_inner_cem<2, 0, 0, KER>;
        case 3: return k_inner_cem<3, 0, 0, KER>;
        case 4: return k_inner_cem<4, 0, 0, KER>;
        case 5: return k_inner_cem<5, 0, 0, KER>;
        case 6: return k_inner_cem<6, 0, 0, KER>;
        case 7: return k_inner_cem<7, 0, 0, KER>;
        case 8: return k_inner_cem<8, 0, 0, KER>;
        case 9: return k_inner_cem<9, 0, 0, KER>;
        case 10: return k_inner_cem<10, 0, 0, KER>;
        default: return nullptr;
    }
}
static inner_cem_fn inner_cem_kernel(const DCfg& d, int kind) {
    return d.kernel == dm::KER_GAUSSIAN ? inner_cem_kernel_k<dm::KER_GAUSSIAN>(d, kind) : inner_cem_kernel_k<dm::KER_LAPLACE>(d, kind);
}
static size_t inner_cem_smem_kind(const DCfg& d, int kind) {
    if (kind == INNER_WARP) return (size_t)warp_layout(d.nr, d.S_in, d.n_el_in).total * sizeof(float);
    if (kind == INNER_CTA || kind == INNER_CTA_LAT || kind == INNER_CTA_FASTMATH) return (size_t)fast_layout(d.nr, d.S_in, d.n_el_in).total * sizeof(float);
    if (kind == INNER_LAT512) return (size_t)(fast_layout(d.nr, d.S_in, d.n_el_in).total + al4(d.S_in) + al4(d.S_in * d.nr) + al4((d.nm + 1) * (d.S_in - d.n_el_in)) + 256) * sizeof(float);
    return (size_t)opt_layout(d.nr, d.np, d.S_in, d.n_el_in).total * sizeof(float);
}

static int create_body(mpcmmd_handle_s* h, const mpcmmd_config* cfg, int device);
extern "C" int mpcmmd_create(const mpcmmd_config* cfg, int device, mpcmmd_handle* out) {
    return mpcmmd_create_with_kernel(cfg, MPCMMD_KERNEL_LAPLACE, device, out);
}
extern "C" int mpcmmd_create_with_kernel(const mpcmmd_config* cfg, int mmd_kernel, int device, mpcmmd_handle* out) {
    if (!cfg || !out) return fail("mpcmmd_create: null argument");
    if (mmd_kernel != MPCMMD_KERNEL_LAPLACE && mmd_kernel != MPCMMD_KERNEL_GAUSSIAN) return fail("mpcmmd_create: mmd_kernel must be 0 (laplace) or 1 (gaussian)");
    if (mmd_kernel == MPCMMD_KERNEL_GAUSSIAN) {
        const char* mode = getenv("MPCMMD_INNER_CEM"); const char* cl = getenv("MPCMMD_CHOL");
        if (mode && (!strcmp(mode, "warp") || !strcmp(mode, "pipe") || !strcmp(mode, "split")))
            return fail("mpcmmd_create: the Gaussian MMD kernel has no MPCMMD_INNER_CEM=warp|pipe|split build (experimental inner-CEM kernels are Laplace only)");
        if (cl && (!strcmp(cl, "la") || !strcmp(cl, "cta")))
            return fail("mpcmmd_create: the Gaussian MMD kernel has no MPCMMD_CHOL=la|cta build (experimental inner-CEM kernels are Laplace only)");
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("mpcmmd_create: no CUDA device (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail("mpcmmd_create: bad device index");
    CK(cudaSetDevice(device));
    const int B = cfg->num_batch, np = cfg->num_prime, nr = cfg->num_reduced, nm = nr * nr, E = cfg->max_episodes;
    if (B < cfg->ellite_num_cost || cfg->ellite_num_cost > 32 || cfg->ellite_num > 8 || cfg->ellite_num > cfg->ellite_num_cost)
        return fail("mpcmmd_create: need ellite_num <= 8, ellite_num <= ellite_num_cost <= min(32, num_batch)");
    if (np < 2 || np > MPCMMD_T) return fail("mpcmmd_create: num_prime must be in [2,100]");
    if (nr < 2 || nr > MPCMMD_MAX_NR_DEV) return fail("mpcmmd_create: num_reduced must be in [2,64] (mmd_opt: 2..40)");
    if (cfg->num_obs < 1 || E < 1) return fail("mpcmmd_create: num_obs and max_episodes must be >= 1");
    if (cfg->num_obs > MPCMMD_MAX_NR_DEV) return fail("mpcmmd_create: num_obs must be <= 64");
    if (cfg->num_samples_cem > RISKO_THREADS * 8 || cfg->num_ellite_beta < 2 || cfg->num_ellite_beta >= cfg->num_samples_cem)
        return fail("mpcmmd_create: bad inner-CEM sizes");
    if (cfg->maxiter_beta_cem < 1 || cfg->maxiter_beta_cem > 64 || cfg->maxiter_beta_cem > SEL_THREADS) return fail("mpcmmd_create: maxiter_beta_cem must be in [1, 64]");
    if (cfg->maxiter_cem < 1 || cfg->maxiter_cem > 4096) return fail("mpcmmd_create: maxiter_cem must be in [1, 4096]");
    if (cfg->ellite_num < 1) return fail("mpcmmd_create: ellite_num must be >= 1");
    if (cfg->noise_kind != 0 && cfg->noise_kind != 1) return fail("mpcmmd_create: noise_kind must be 0 (gaussian) or 1 (beta)");
    if (B < 1 || B > (1 << 20)) return fail("mpcmmd_create: num_batch must be in [1, 2^20]");
    mpcmmd_handle_s* h = new mpcmmd_handle_s();
    h->device = device; h->cfg = *cfg; h->E = E; h->d.kernel = mmd_kernel;
    if (create_body(h, cfg, device)) { mpcmmd_destroy(h); return -1; }      // one cleanup path: every failure after the allocation frees the handle and its device memory
    *out = h;
    return 0;
}
static int create_body(mpcmmd_handle_s* h, const mpcmmd_config* cfg, int device) {
    const int B = cfg->num_batch, np = cfg->num_prime, nr = cfg->num_reduced, nm = nr * nr, E = cfg->max_episodes;
    DCfg& d = h->d;
    d.B = B; d.np = np; d.nr = nr; d.nm = nm; d.O = cfg->num_obs; d.iters = cfg->maxiter_cem; d.n_el = cfg->ellite_num;
    d.n_el_cost = cfg->ellite_num_cost; d.noise_kind = cfg->noise_kind; d.S_in = cfg->num_samples_cem; d.iters_in = cfg->maxiter_beta_cem;
    d.n_el_in = cfg->num_ellite_beta;
    d.sigma_acc = cfg->sigma_acc; d.sigma_steer = cfg->sigma_steer; d.ksig_steer = cfg->ksig_steer; d.acc_const = cfg->acc_const_noise;
    d.steer_const = cfg->steer_const_noise; d.beta_a = cfg->beta_a; d.beta_b = cfg->beta_b;
    d.v_min = cfg->v_min; d.v_max = cfg->v_max; d.a_max = cfg->a_max;
    d.b_lane_ub = 1.0f * cfg->y_ub; d.b_lane_lb = -1.0f * cfg->y_lb;         // projection.py:127-128, gamma = 1
    d.y_lb = cfg->y_lb; d.y_ub = cfg->y_ub; d.a2_obs = cfg->a_obs_sq; d.b2_obs = cfg->b_obs_sq;
    d.wheel_base = cfg->wheel_base; d.dt = cfg->dt; d.steer_max = cfg->steer_max; d.steer_rate_pen = cfg->steer_rate_pen;
    d.alpha_quant = cfg->alpha_quant; d.ker_wt = cfg->ker_wt; d.lam_inv = cfg->lamda_inv;
    d.one_m_alpha_mean = cfg->one_minus_alpha_mean; d.alpha_mean = cfg->alpha_mean;
    d.one_m_alpha_cov = cfg->one_minus_alpha_cov; d.alpha_cov = cfg->alpha_cov;
    d.sigma_clip = cfg->sigma_clip; d.inv_nm = (float)(1.0 / nm); d.m2_inv_nm = (float)(-2.0 * (1.0 / nm)); d.beta_del = (float)(1.0 / nr);
    d.sigma_random = cfg->sigma_random;
    d.obs_win = (float)(sqrt((double)cfg->a_obs_sq) * (1.0 + 1e-6) + 1.0e-2);
#define UP(dst, src, n) if (upload(h, &d.dst, cfg->src, (n))) return -1;
    UP(Wfit, Wfit, (size_t)NV * np)
#undef UP
    {   // P | Pd | Pdd | Gx | Gy | Kx | Ky in one block (cudaMalloc: 256-byte aligned), the layout k_project's shared memory mirrors
        const float* src[7] = {cfg->P, cfg->Pdot, cfg->Pddot, cfg->Gx, cfg->Gy, cfg->Kx, cfg->Ky};
        const int cnt[7] = {1100, 1100, 1100, 77, 88, 154, 165};
        std::vector<float> blk; blk.reserve(PROJ_CONST_FLOATS);
        for (int i = 0; i < 7; i++) { if (!src[i]) return fail("mpcmmd_create: null matrix pointer in config"); blk.insert(blk.end(), src[i], src[i] + cnt[i]); }
        const float* base = nullptr;
        if ((int)blk.size() != PROJ_CONST_FLOATS || upload(h, &base, blk.data(), blk.size())) return -1;
        d.proj_const = base; d.P = base; d.Pd = base + 1100; d.Pdd = base + 2200; d.Gx = base + 3300; d.Gy = d.Gx + 77; d.Kx = d.Gy + 88; d.Ky = d.Kx + 154;
    }
    {   // operands of k_project_tc: each Bernstein matrix as a [4 chunks][112 knots][4 coefficients] image, split x = hi + lo into two
        // tf32 values (round to nearest, ties away: cvt.rna.tf32.f32), followed by Gx | Gy | Kx | Ky
        auto rna = [](float x) { uint32_t u; memcpy(&u, &x, 4); u = (u + 0x1000u) & 0xFFFFE000u; float r; memcpy(&r, &u, 4); return r; };
        std::vector<float> img(ptc::CONST_BYTES / 4, 0.0f);
        const float* mats[3] = {cfg->P, cfg->Pdot, cfg->Pddot};
        for (int m = 0; m < 3; m++)
            for (int t = 0; t < T_; t++)
                for (int j = 0; j < NV; j++) {
                    const float x = mats[m][t * NV + j], hi = rna(x), lo = rna(x - hi);
                    const size_t off = (size_t)(j / 4) * (ptc::KSTR / 4) + (size_t)t * 4 + (j % 4);
                    img[(size_t)(2 * m) * (ptc::IMG / 4) + off] = hi;
                    img[(size_t)(2 * m + 1) * (ptc::IMG / 4) + off] = lo;
                    const size_t offr = (size_t)(t / 4) * (ptc::RSTR / 4) + (size_t)j * 4 + (t % 4);      // transposed: [4-knot chunk][coefficient][knot]
                    img[ptc::OFF_R / 4 + (size_t)(2 * m) * (ptc::RIMG / 4) + offr] = hi;
                    img[ptc::OFF_R / 4 + (size_t)(2 * m + 1) * (ptc::RIMG / 4) + offr] = lo;
                }
        size_t o = ptc::B_BYTES / 4;
        const float* sm[4] = {cfg->Gx, cfg->Gy, cfg->Kx, cfg->Ky}; const int cnt[4] = {77, 88, 154, 165};
        for (int i = 0; i < 4; i++) { memcpy(&img[o], sm[i], cnt[i] * sizeof(float)); o += cnt[i]; }
        for (int m = 0; m < 3; m++) { memcpy(&img[o], mats[m], NV * sizeof(float)); o += NV; }     // fp32 rows of knot 0
        if (upload(h, &d.proj_tc_const, img.data(), img.size())) return -1;
        const char* pv = getenv("MPCMMD_PROJ");               // "tc": tensor-core projection (tolerance parity, see k_project_tc.cuh)
        h->proj_tc = pv && (!strcmp(pv, "tc") || !strcmp(pv, "tc-always"));
        h->proj_tc_always = pv && !strcmp(pv, "tc-always");   // tests / probes: every launch, whatever its size
    }
    DWork& w = h->w;
    const size_t EB = (size_t)E * B, n = (size_t)nr * np, ncem = (size_t)(B - d.n_el) * NPAR;
#define AL(p, cnt) if (dalloc(h, &w.p, (cnt))) return -1;
    AL(params, EB * NPAR) AL(lam_x, EB * NV) AL(lam_y, EB * NV) AL(s_lane, EB * 2 * NL) AL(mean, (size_t)E * NPAR) AL(cov, (size_t)E * 64)
    AL(cx, EB * NV) AL(cy, EB * NV) AL(res_norm, EB) AL(cost_base, EB) AL(acc, EB * T_) AL(steer, EB * T_) AL(risk, EB) AL(lane, EB)
    AL(beta, EB * nr) AL(sigma, EB) AL(res_beta, EB * d.iters_in)
    AL(z1, (size_t)E * d.iters * n) AL(z2, (size_t)E * d.iters * n) AL(z3, (size_t)E * d.iters * n) AL(zcem, (size_t)E * d.iters * ncem)
    AL(keys, (size_t)E * d.iters * 4)
    if (d.noise_kind == 1) { AL(btab, (size_t)E * d.iters * 4 * GT_FIELDS * n) } else w.btab = nullptr;
    AL(idx_mpc, E) AL(init_state, (size_t)E * 6) AL(mean0, (size_t)E * NPAR) AL(cov0, (size_t)E * 64)
    AL(x_obs, (size_t)E * d.O * T_) AL(y_obs, (size_t)E * d.O * T_) AL(v_des, E)
    if (d.O > OBS_SORT_MIN) { AL(sx_obs, (size_t)E * d.O * T_) AL(sy_obs, (size_t)E * d.O * T_) AL(obs_nan, (size_t)E * T_) } else { w.sx_obs = w.sy_obs = nullptr; w.obs_nan = nullptr; }
    AL(o_cx, (size_t)E * NV) AL(o_cy, (size_t)E * NV) AL(o_lane, E) AL(o_obs, E) AL(o_beta, (size_t)E * nr) AL(o_sigma, E)
    AL(o_res_beta, (size_t)E * d.iters_in) AL(o_sel, (size_t)E * d.iters)
#undef AL
    if (dalloc(h, &h->beq_x, (size_t)E * 3) || dalloc(h, &h->beq_y, (size_t)E * 4) || dalloc(h, &h->state0, (size_t)E * 5)) return -1;
    // constant normal tables [survey Q8]: every key below derives from PRNGKey(0) only
    {
        const int S = d.S_in, dd = nm + 1, ne = d.n_el_in;
        float *z_init, *theta0, *zb, *ztmp;
        if (dalloc(h, &z_init, (size_t)B * NPAR) || dalloc(h, &theta0, (size_t)S * dd) || dalloc(h, &zb, (size_t)d.iters_in * (S - ne) * dd) ||
            dalloc(h, &ztmp, (size_t)S * dd)) return -1;
        // host-side key derivation mirrors the device functions (integer-only Threefry)
        auto tf = [](uint32_t k0, uint32_t k1, uint32_t x0, uint32_t x1, uint32_t* o) {
            auto rotl = [](uint32_t x, int r) { return (x << r) | (x >> (32 - r)); };
            const int R[2][4] = {{13, 15, 26, 6}, {17, 29, 16, 24}};
            uint32_t ks[3] = {k0, k1, k0 ^ k1 ^ 0x1BD11BDAu};
            x0 += ks[0]; x1 += ks[1];
            for (int i = 0; i < 5; i++) {
                for (int r = 0; r < 4; r++) { x0 += x1; x1 = rotl(x1, R[i & 1][r]); x1 ^= x0; }
                x0 += ks[(i + 1) % 3]; x1 += ks[(i + 2) % 3] + (uint32_t)(i + 1);
            }
            o[0] = x0; o[1] = x1;
        };
        auto split0 = [&](uint32_t* k) { uint32_t a[2], b[2]; tf(k[0], k[1], 0u, 2u, a); tf(k[0], k[1], 1u, 3u, b); k[0] = a[0]; k[1] = b[0]; };
        uint32_t key_init[2] = {0u, 0u};
        split0(key_init);                                                         // cem_helper.py:125 / compute_beta.py:108
        k_normal_table<<<64, 256>>>(key_init[0], key_init[1], B * NPAR, z_init);
        uint32_t kk[2] = {key_init[0], key_init[1]};
        split0(kk);                                                               // compute_beta.py:44
        k_normal_table<<<64, 256>>>(kk[0], kk[1], S * dd, ztmp);
        k_theta0<<<64, 256>>>(ztmp, S, dd, d.sigma_clip, theta0);
        uint32_t carry[2] = {key_init[0], key_init[1]};
        for (int it = 0; it < d.iters_in; it++) {
            split0(carry);                                                        // compute_beta.py:131
            uint32_t dk[2] = {carry[0], carry[1]};
            split0(dk);                                                           // compute_beta.py:54
            k_normal_table<<<64, 256>>>(dk[0], dk[1], (S - ne) * dd, zb + (size_t)it * (S - ne) * dd);
        }
        float* zbT;
        if (dalloc(h, &zbT, (size_t)d.iters_in * (S - ne) * dd)) return -1;
        k_transpose_tables<<<64, 256>>>(zb, zbT, d.iters_in, S - ne, dd);
        float* th0T;
        if (dalloc(h, &th0T, (size_t)S * dd)) return -1;
        k_transpose_tables<<<64, 256>>>(theta0, th0T, 1, S, dd);
        d.z_init = z_init; d.theta0 = theta0; d.theta0T = th0T; d.zb_iter = zb; d.zb_iterT = zbT;
    }
    // opt-in shared memory sizes (raise-only per (device, kernel): see raise_smem)
    cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device);
    if (h->sm_count < 1) h->sm_count = 1;
    if (raise_smem(device, (const void*)k_project, PROJ_SMEM_BYTES)) return fail("k_project smem opt-in failed");
    if (raise_smem(device, (const void*)k_project_tc, ptc::SMEM_BYTES, true)) return fail("k_project_tc smem opt-in failed");
    {
        size_t rs = nr <= MPCMMD_MAX_NR_OPT ? roll_smem(h, MPCMMD_COST_MMD_OPT) : 0; const size_t rb = roll_smem(h, MPCMMD_COST_CVAR); if (rb > rs) rs = rb;
        if (rs > 227 * 1024) return fail("mpcmmd_create: rollouts of one sample do not fit in shared memory");
        for (int mode = 0; mode < 3; mode++) for (int nz = 0; nz < 3; nz++) for (int so = 0; so < 2; so++) for (int ov = 0; ov < 3; ov++) {
            const void* f = rollouts_kernel(mode, nz, so, ov);
            if (f && raise_smem(device, f, rs)) return fail("k_rollouts smem opt-in failed");
        }
    }
    {
        const char* mode = getenv("MPCMMD_INNER_CEM");       // test / profiling override of the kernel choice
        h->inner_mode = !mode ? 0 : !strcmp(mode, "warp") ? INNER_WARP : !strcmp(mode, "cta") ? INNER_CTA : !strcmp(mode, "generic") ? INNER_GENERIC :
                        !strcmp(mode, "lat") ? INNER_CTA_LAT : !strcmp(mode, "split") ? INNER_SPLIT : !strcmp(mode, "pipe") ? INNER_PIPE : !strcmp(mode, "lat512") ? INNER_LAT512 : 0;
        if (!inner_cem_is_fast(d) && h->inner_mode != 0) h->inner_mode = INNER_GENERIC;
        if (inner_cem_is_fast(d)) {
            const SplitKernels sk = split_kernels(d.nr);
            if (raise_smem(device, (const void*)sk.eval, split_eval_smem(d)) || raise_smem(device, (const void*)sk.update, split_update_smem(d), true))
                return fail("k_icem smem opt-in failed");
            cudaFuncSetAttribute(sk.eval, cudaFuncAttributePreferredSharedMemoryCarveout, 50);     // 12 CTAs x 5.5 KB of operands, the rest stays L1
            const char* mb = getenv("MPCMMD_PIPE_MINB");
            if (mb) h->pipe_minb = atoi(mb);
            if (raise_smem(device, (const void*)pipe_kernel(d.nr, h->pipe_minb), pipe_smem_bytes(d.nr, d.S_in, d.n_el_in), true)) return fail("k_inner_cem_pipe smem opt-in failed");
        }
        { const char* mm = getenv("MPCMMD_MATH"); h->fast_math = mm && !strcmp(mm, "fast"); }
        { const char* cl = getenv("MPCMMD_CHOL"); g_chol = !cl ? 0 : !strcmp(cl, "la") ? 1 : !strcmp(cl, "cta") ? 2 : 0; }
        for (int kind = INNER_WARP; kind <= INNER_LAT512; kind++) {
            if (kind == INNER_SPLIT || kind == INNER_PIPE || kind == INNER_BIG) continue;
            if (kind != INNER_GENERIC && !inner_cem_is_fast(d)) continue;
            inner_cem_fn f = inner_cem_kernel(d, kind);
            if (!f) continue;
            const size_t sm = inner_cem_smem_kind(d, kind);
            if (sm > 227 * 1024) return fail("mpcmmd_create: reduced-set state does not fit in shared memory");
            if (raise_smem(device, (const void*)f, sm, kind != INNER_GENERIC)) return fail("k_inner_cem smem opt-in failed");
            if (kind == INNER_WARP) {
                int per_sm = 0;
                if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, f, 32, sm) != cudaSuccess || per_sm < 1) per_sm = 1;
                h->warp_grid = per_sm * h->sm_count;
            }
        }
    }
    CK(cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming));
    for (int i = 0; i < MAX_GROUPS - 1; i++) {
        CK(cudaStreamCreateWithFlags(&h->aux_stream[i], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&h->ev_join[i], cudaEventDisableTiming));
    }
    { const char* gv = getenv("MPCMMD_GROUPS"); h->groups_override = gv ? atoi(gv) : 0; }
    { const char* pv = getenv("MPCMMD_PRIO"); h->prio_mode = pv ? atoi(pv) : 0; }
    {   // MPCMMD_CARVE=1 (experiment): every kernel of a solve prefers the maximum shared-memory carve-out, so that kernels of concurrent branches / handles
        // never wait for an SM to drain before its L1 / shared split can change
        const char* cv = getenv("MPCMMD_CARVE");
        if (cv) {
            const void* fns[] = {(const void*)k_project, rollouts_kernel(ROLL_OPT, NZ_BETA_TABLE, 0), rollouts_kernel(ROLL_FLY, NZ_BETA_TABLE, 0), rollouts_kernel(ROLL_STAGED, NZ_BETA_TABLE, 0),
                                 (const void*)k_opt_risk<false>, (const void*)k_select, (const void*)k_noise, (const void*)k_init, (const void*)k_boundary};
            for (const void* f : fns) cudaFuncSetAttribute(f, cudaFuncAttributePreferredSharedMemoryCarveout, atoi(cv) == 1 ? cudaSharedmemCarveoutMaxShared : cudaSharedmemCarveoutDefault);
        }
    }
    CK(cudaDeviceSynchronize());
    CK(cudaGetLastError());
    return 0;
}

extern "C" int mpcmmd_destroy(mpcmmd_handle h) {
    if (!h) return 0;
    cudaSetDevice(h->device);
    for (auto& g : h->graphs) cudaGraphExecDestroy(g.second);
    for (void* p : h->allocs) cudaFree(p);
    if (h->own_stream) cudaStreamDestroy(h->own_stream);
    for (int i = 0; i < MAX_GROUPS - 1; i++) { if (h->aux_stream[i]) cudaStreamDestroy(h->aux_stream[i]); if (h->ev_join[i]) cudaEventDestroy(h->ev_join[i]); }
    if (h->ev_fork) cudaEventDestroy(h->ev_fork);
    delete h;
    return 0;
}

static size_t sel_smem(const DCfg& d) { return d.B <= SEL_RANK_MAX ? 2 * (size_t)d.B * sizeof(float) : 16; }
static float w_obs_for(const mpcmmd_handle_s* h, int kind) { (void)h; return kind == MPCMMD_COST_SAA ? 1.0e6f : 1.0e3f; }   // cem.py:161-163

static ProjArgs proj_args(mpcmmd_handle_s* h, int n_ep) {
    ProjArgs p;
    p.n_samples = n_ep * h->d.B; p.B = h->d.B; p.params = h->w.params; p.beq_x = h->beq_x; p.beq_y = h->beq_y; p.v_des = h->w.v_des;
    p.lam_x = h->w.lam_x; p.lam_y = h->w.lam_y; p.s_lane = h->w.s_lane; p.cx = h->w.cx; p.cy = h->w.cy; p.res_norm = h->w.res_norm;
    p.cost_base = h->w.cost_base; p.acc = h->w.acc; p.steer = h->w.steer; p.dbg = 0;
    return p;
}
static int launch_project(mpcmmd_handle_s* h, const ProjArgs& p, cudaStream_t s) {
    // MPCMMD_PROJ=tc: the tensor-core kernel for throughput-sized launches.  One of its CTAs walks the 100 knots of 128 samples serially
    // (~115 us alone on an SM, measured), so small launches (latency regime, e.g. one episode = 100 samples: 29 us) keep the warp-per-sample kernel.
    if (h->proj_tc && (h->proj_tc_always || p.n_samples >= 64 * h->sm_count)) {
        k_project_tc<<<(p.n_samples + ptc::THREADS - 1) / ptc::THREADS, ptc::CTA_THREADS, ptc::SMEM_BYTES, s>>>(h->d, p);
        return 0;
    }
    const int blocks = (p.n_samples + PROJ_WARPS - 1) / PROJ_WARPS;
    k_project<<<blocks, PROJ_WARPS * 32, PROJ_SMEM_BYTES, s>>>(h->d, p);
    return 0;
}
// mother rollouts / features scratch of the mmd_opt path, allocated on first use ([E*B][nm][np] x2 and [E*B][nm][22])
static int ensure_opt_scratch(mpcmmd_handle_s* h) {
    if (h->xroll) return 0;
    if (h->d.nr > MPCMMD_MAX_NR_OPT) return fail("mmd_opt: num_reduced must be in [2, 40] (larger reduced sets: cvar / saa / mmd_random only)");
    const DCfg& d = h->d; const size_t EB = (size_t)h->E * d.B;
    if (d.nr > MPCMMD_MAX_NR) {      // large reduced sets: chain state in global memory, as many chains at a time as the scratch budget holds
        const size_t per = big_layout(d.nr, d.S_in, d.n_el_in).total * sizeof(float);
        size_t chunk = MPCMMD_BIG_SCRATCH_BYTES / per; if (chunk < 1) chunk = 1; if (chunk > EB) chunk = EB;
        h->big_chunk = (int)chunk;
        if (dalloc(h, &h->big_state, chunk * (per / sizeof(float)))) return -1;
    }
    if (dalloc(h, &h->feat, EB * d.nm * 2 * NV) || dalloc(h, &h->ctrl, EB * 2 * d.nr * d.np)) return -1;
    // the mother rollouts are stored only for the kernels that read them back (generic / warp-per-chain); allocated on first such launch
    h->xroll = h->feat;     // non-null marker: scratch is ready
    if (!inner_cem_is_fast(d) || h->inner_mode == INNER_WARP || h->inner_mode == INNER_GENERIC) {
        if (dalloc(h, &h->rolls_x, EB * d.nm * d.np) || dalloc(h, &h->rolls_y, EB * d.nm * d.np)) return -1;
    }
    if (dalloc(h, &h->ridx, EB * d.nr)) return -1;
    if (inner_cem_is_fast(d) && dalloc(h, &h->bscratch, EB * d.S_in * (d.nr + 1))) return -1;
    if (inner_cem_is_fast(d) && dalloc(h, &h->mrisk, EB * d.nm * 3)) return -1;
    // scratch of the opt-in variants only when they are selected (0.35 GB at 200 episodes)
    if (inner_cem_is_fast(d) && h->inner_mode == INNER_PIPE && dalloc(h, &h->throws, EB * (d.nm + 1) * ICP_TH_LD)) return -1;
    if (inner_cem_is_fast(d) && h->inner_mode == INNER_SPLIT && dalloc(h, &h->split_state, EB * split_layout(d.nr, d.S_in, d.n_el_in).total)) return -1;
    if (inner_cem_is_fast(d) && h->warp_grid > 0 && dalloc(h, &h->stash, (size_t)h->warp_grid * d.S_in * ICW_STASH_LD)) return -1;
    CK(cudaDeviceSynchronize());     // dalloc's memsets run on the legacy default stream; solves run on non-blocking streams that do not wait for it
    return 0;
}
// rollouts (+ risk for the num_reduced-rollout costs); mmd_opt continues with the inner CEM kernel.  Returns launches issued.
static int launch_risk(mpcmmd_handle_s* h, const RiskArgs& r, cudaStream_t s, int* n_launch = nullptr) {
    const DCfg& d = h->d;
    const bool opt = r.cost_kind == MPCMMD_COST_MMD_OPT;
    if (r.n_samples > h->E * d.B) return fail("risk stage: more samples than the workspace holds (max_episodes * num_batch)");
    RollArgs ra;
    ra.r = r; ra.spb = roll_spb(h, r.cost_kind, r.n_samples); ra.R = opt ? d.nm : d.nr; ra.xroll = h->xroll; ra.yroll = h->yroll; ra.feat = h->feat; ra.stash = nullptr; ra.ridx = h->ridx; ra.bscratch = h->bscratch; ra.ctrl = h->ctrl; ra.write_rolls = 0; ra.fold_risk = 0; ra.mrisk = h->mrisk; ra.stage_ctrl = roll_stage_ctrl(h, r.cost_kind, r.n_samples);
    inner_cem_fn f = nullptr;
    int kind = INNER_GENERIC;
    if (opt) {
        // default: one 3-warp CTA per chain (k_inner_cem_fast).  The warp-per-chain persistent kernel is kept as an opt-in
        // (MPCMMD_INNER_CEM=warp): measured 233 ms vs 209 ms per 200-episode mmd_opt solve on B200 (profiles/r01_v7_summary.md) --
        // 19 independent instruction streams per SM thrash the 32 KB instruction cache.
        // a launch that fits in one wave of resident CTAs (e.g. a single episode) is latency-bound: take the build with the 96-register budget
        // a launch of at most 3 chains per SM (one episode = 100 chains) is pure dependency latency: the latency build of the fused kernel
        // (at most one chain per SM: the 16-warp latency kernel k_inner_cem_lat; up to 3 per SM: the 3-warp latency build of the fused kernel)
        if (inner_cem_is_fast(d)) kind = h->inner_mode ? h->inner_mode : (r.n_samples <= h->sm_count ? INNER_LAT512 : r.n_samples <= 3 * h->sm_count ? INNER_CTA_LAT : INNER_DEFAULT_THROUGHPUT);
        if (d.nr > MPCMMD_MAX_NR) kind = INNER_BIG;
        if (kind == INNER_PIPE && !pipe_ok(d)) kind = INNER_CTA;
        if (kind == INNER_CTA && h->fast_math) kind = INNER_CTA_FASTMATH;
        if (kind == INNER_WARP && !h->stash) return fail("internal: row stash of k_inner_cem_warp not allocated");
        if (kind != INNER_SPLIT && kind != INNER_PIPE && kind != INNER_BIG) {
            f = inner_cem_kernel(d, kind);
            if (!f) return fail("mmd_opt: num_reduced must be in [2, 10]");
        }
        if (!h->xroll) return fail("internal: mmd_opt scratch not allocated");
        ra.stash = h->stash;
        // latency regime (at most 3 chains per SM): the serial rollout recurrence is the cost of every kernel, so k_opt_risk's re-roll of the chosen reduced set is
        // replaced by maxima the mother rollouts fold in themselves (mmd_opt p50 at batch 1: 6.79 -> 6.57 ms).  Larger launches keep the re-roll: the extra
        // obstacle work in k_rollouts (+20 %) costs more than the short k_opt_risk it removes (measured at 13 / 25 / 50 episodes: 14.4 / 22.9 / 41.8 ms vs 14.7 / 24.0 / 42.4)
        if (kind != INNER_GENERIC && kind != INNER_WARP && kind != INNER_BIG && h->mrisk && d.O <= OBS_SORT_MIN && r.n_samples <= 3 * h->sm_count) ra.fold_risk = 1;
        if (kind != INNER_CTA && kind != INNER_CTA_LAT && kind != INNER_CTA_FASTMATH && kind != INNER_LAT512 && kind != INNER_SPLIT && kind != INNER_PIPE) {          // these kernels evaluate the risk themselves from the stored mother rollouts
            if (!h->rolls_x) return fail("internal: mother-rollout scratch not allocated");
            ra.write_rolls = 1; ra.xroll = h->rolls_x; ra.yroll = h->rolls_y;
        }
    }
    {
        if (ra.fold_risk) ra.spb = 1;
        const int grid = (r.n_samples + ra.spb - 1) / ra.spb; const size_t rsm = roll_smem_for(d, r.cost_kind, ra.spb, ra.stage_ctrl, ra.fold_risk);
        const int nz = d.noise_kind == 0 ? NZ_GAUSS : (r.btab && !r.binj1) ? NZ_BETA_TABLE : NZ_ANY;
        const int mode = opt ? ROLL_OPT : ra.stage_ctrl ? ROLL_STAGED : ROLL_FLY;
        const void* fk = rollouts_kernel(mode, nz, mode == ROLL_FLY && r.sx_obs, ra.fold_risk ? OV_FOLD : ra.write_rolls ? OV_WRITE : OV_PLAIN);
        void* kargs[] = {(void*)&d, (void*)&ra};
        CK(cudaLaunchKernel(fk, dim3(grid), dim3(ROLL_THREADS), kargs, rsm, s));
    }
    if (n_launch) *n_launch = 1;
    if (opt && kind == INNER_BIG) {
        if (!h->big_state) return fail("internal: large-reduced-set scratch not allocated");
        int nl = 1;
        for (int g0 = 0; g0 < r.n_samples; g0 += h->big_chunk) {       // chain ranges share the scratch: launches on one stream run in order
            const int nc = r.n_samples - g0 < h->big_chunk ? r.n_samples - g0 : h->big_chunk;
            const bool gauss = d.kernel == dm::KER_GAUSSIAN;
            if (r.n_samples <= h->sm_count) (gauss ? k_inner_cem_big<BIG_THREADS, dm::KER_GAUSSIAN> : k_inner_cem_big<BIG_THREADS>)<<<nc, BIG_THREADS, 0, s>>>(d, ra, h->big_state, g0, nc);
            else (gauss ? k_inner_cem_big<BIG_THREADS_SMALL, dm::KER_GAUSSIAN> : k_inner_cem_big<BIG_THREADS_SMALL>)<<<nc, BIG_THREADS_SMALL, 0, s>>>(d, ra, h->big_state, g0, nc);
            nl++;
        }
        if (n_launch) *n_launch = nl;
    } else if (opt && kind == INNER_PIPE) {
        pipe_kernel(d.nr, h->pipe_minb)<<<(r.n_samples + 1) / 2, ICP_THREADS, pipe_smem_bytes(d.nr, d.S_in, d.n_el_in), s>>>(d, ra, h->throws);
        { const int ospb = OPT_RISK_THREADS / d.nr; if (r.sx_obs) k_opt_risk<true><<<(r.n_samples + ospb - 1) / ospb, OPT_RISK_THREADS, 0, s>>>(d, ra); else k_opt_risk<false><<<(r.n_samples + ospb - 1) / ospb, OPT_RISK_THREADS, 0, s>>>(d, ra); }
        if (n_launch) *n_launch = 3;
    } else if (opt && kind == INNER_SPLIT) {
        const SplitKernels sk = split_kernels(d.nr);
        SplitArgs sa;
        sa.n_chains = r.n_samples; sa.g0 = 0; sa.state = h->split_state; sa.feat = h->feat; sa.bscratch = h->bscratch;
        sa.beta = r.beta; sa.sigma = r.sigma; sa.res_beta = r.res_beta; sa.ridx = h->ridx;
        const long long nd = (long long)r.n_samples * d.nm * d.nm;
        sk.dist<<<(unsigned)((nd + 255) / 256), 256, 0, s>>>(d, sa);
        const size_t se = split_eval_smem(d), su = split_update_smem(d);
        for (int it = 0; it < d.iters_in; it++) {
            sk.eval<<<r.n_samples, (it == 0 && d.S_in > ICE_THREADS) ? 128 : ICE_THREADS, se, s>>>(d, sa, it);
            sk.update<<<(r.n_samples + ICU_WARPS - 1) / ICU_WARPS, ICU_WARPS * 32, su, s>>>(d, sa, it);
        }
        { const int ospb = OPT_RISK_THREADS / d.nr; if (r.sx_obs) k_opt_risk<true><<<(r.n_samples + ospb - 1) / ospb, OPT_RISK_THREADS, 0, s>>>(d, ra); else k_opt_risk<false><<<(r.n_samples + ospb - 1) / ospb, OPT_RISK_THREADS, 0, s>>>(d, ra); }
        if (n_launch) *n_launch = 3 + 2 * d.iters_in;
    } else if (opt) {
        const size_t sm = inner_cem_smem_kind(d, kind);
        if (kind == INNER_WARP) f<<<r.n_samples < h->warp_grid ? r.n_samples : h->warp_grid, 32, sm, s>>>(d, ra);
        else f<<<r.n_samples, kind == INNER_LAT512 ? ICL_THREADS : (kind == INNER_CTA || kind == INNER_CTA_LAT || kind == INNER_CTA_FASTMATH) ? ICF_THREADS : risko_threads(d.nr), sm, s>>>(d, ra);
        if (n_launch) *n_launch = 2;
        if (kind == INNER_CTA || kind == INNER_CTA_LAT || kind == INNER_CTA_FASTMATH || kind == INNER_LAT512) {
            { const int ospb = OPT_RISK_THREADS / d.nr; if (r.sx_obs) k_opt_risk<true><<<(r.n_samples + ospb - 1) / ospb, OPT_RISK_THREADS, 0, s>>>(d, ra); else k_opt_risk<false><<<(r.n_samples + ospb - 1) / ospb, OPT_RISK_THREADS, 0, s>>>(d, ra); }
            if (n_launch) *n_launch = 3;
        }
    }
    return 0;
}

// enqueue the whole solve on `s` (captured into a graph by the caller)
// `marks` (optional, profiling only): an event is recorded after every launch, tagged with its kernel class
struct LaunchMark { cudaEvent_t ev; int cls; };      // cls: 0 setup (boundary/noise/init), 1 project, 2 risk, 3 select
static int enqueue_solve(mpcmmd_handle_s* h, int kind, int n_ep, cudaStream_t s, int* launches, std::vector<LaunchMark>* marks = nullptr) {
    const DCfg& d = h->d; DWork& w = h->w;
    const size_t n = (size_t)d.nr * d.np, ncem = (size_t)(d.B - d.n_el) * NPAR;
    int cnt = 0;
    auto mark = [&](int cls) { cnt++; if (marks) { LaunchMark m; cudaEventCreate(&m.ev); cudaEventRecord(m.ev, s); m.cls = cls; marks->push_back(m); } };
    k_boundary<<<(n_ep + 127) / 128, 128, 0, s>>>(w.init_state, h->beq_x, h->beq_y, h->state0, n_ep); mark(0);
    if (w.sx_obs) { k_obs_sort<<<(n_ep * T_ + 127) / 128, 128, 0, s>>>(w.x_obs, w.y_obs, w.sx_obs, w.sy_obs, w.obs_nan, d.O, n_ep * T_); mark(0); }
    k_noise<<<n_ep * d.iters, d.B <= SEL_RANK_MAX ? 128 : 1024, 0, s>>>(d, w, n_ep, 0, d.iters); mark(0);
    k_init<<<n_ep, d.B <= SEL_RANK_MAX ? 128 : 1024, 0, s>>>(d, w, n_ep); mark(0);
    for (int it = 0; it < d.iters; it++) {
        ProjArgs p = proj_args(h, n_ep);
        launch_project(h, p, s); mark(1);
        RiskArgs r;
        r.n_samples = n_ep * d.B; r.B = d.B; r.cost_kind = kind; r.acc = w.acc; r.steer = w.steer; r.state0 = h->state0;
        r.z1 = w.z1 + it * n; r.z2 = w.z2 + it * n; r.z3 = w.z3 + it * n; r.z_stride = (size_t)d.iters * n;
        r.keys = w.keys + it * 4; r.key_stride = (size_t)d.iters * 4;
        r.btab = w.btab ? w.btab + (size_t)it * 4 * GT_FIELDS * n : nullptr; r.btab_stride = (size_t)d.iters * 4 * GT_FIELDS * n; r.binj1 = r.binj2 = nullptr;
        r.x_obs = w.x_obs; r.y_obs = w.y_obs; r.sx_obs = w.sx_obs; r.sy_obs = w.sy_obs; r.obs_nan = w.obs_nan; r.risk = w.risk; r.lane = w.lane; r.beta = w.beta; r.sigma = w.sigma; r.res_beta = w.res_beta;
        int nl = 0;
        if (launch_risk(h, r, s, &nl)) return -1;
        mark(2); cnt += nl - 1;
        SelArgs a;
        a.n_ep = n_ep; a.B = d.B; a.it = it; a.nr = d.nr; a.iters_in = d.iters_in; a.w_obs = w_obs_for(h, kind);
        a.res_norm = w.res_norm; a.risk = w.risk; a.lane = w.lane; a.cost_base = w.cost_base; a.params = w.params; a.mean = w.mean; a.cov = w.cov;
        a.zcem = w.zcem + it * ncem; a.z_stride = (size_t)d.iters * ncem; a.cx = w.cx; a.cy = w.cy; a.beta = w.beta; a.sigma = w.sigma;
        a.res_beta = w.res_beta; a.o_cx = w.o_cx; a.o_cy = w.o_cy; a.o_lane = w.o_lane; a.o_obs = w.o_obs; a.o_beta = w.o_beta;
        a.o_sigma = w.o_sigma; a.o_res_beta = w.o_res_beta; a.o_sel = w.o_sel; a.sel_stride = d.iters;
        k_select<<<n_ep, d.B <= SEL_RANK_MAX ? SEL_THREADS : SEL_THREADS_BIG, sel_smem(d), s>>>(d, a); mark(3);
    }
    *launches = cnt;
    return 0;
}

// number of episode groups (branches) of a solve graph.  Groups pay off for mmd_opt launches of a few waves of chains (strong-scaled shards: 25 episodes = 2500
// chains on 1776 resident CTAs): the groups drift out of phase, so one group's tail wave and small kernels are filled by the others' chains.  Measured
// (tools/overlap_probe.py, mmd_opt solve of 25 / 50 / 100 episodes): 1 group 24.2 / 41.9 / 78.8 ms, 2 groups 22.6 / 41.1 / 79.5, 3 groups 21.6 / 39.9 / 78.2,
// 4 groups 22.5 / 42.9 / 78.4.
static int solve_groups(const mpcmmd_handle_s* h, int kind, int n_ep) {
    if (n_ep < 2 || h->inner_mode == INNER_WARP) return 1;         // the warp-per-chain kernel's row stash is per persistent CTA, not per chain
    if (h->groups_override >= 1 && h->groups_override <= MAX_GROUPS) return h->groups_override < n_ep ? h->groups_override : n_ep;
    const long long chains = (long long)n_ep * h->d.B;
    if (kind != MPCMMD_COST_MMD_OPT || !inner_cem_is_fast(h->d) || chains <= 6LL * h->sm_count || chains > 36LL * h->sm_count) return 1;
    const int G = chains > 12LL * h->sm_count ? 3 : 2;
    return G < n_ep ? G : n_ep;              // never an empty group (large num_batch: few episodes, many chains)
}
static int get_graph(mpcmmd_handle_s* h, int kind, int n_ep, cudaGraphExec_t* out) {
    auto key = std::make_pair(kind, n_ep);
    auto it = h->graphs.find(key);
    if (it != h->graphs.end()) { *out = it->second; h->last_launches = h->graph_launches[key]; return 0; }
    cudaGraph_t g;
    int launches = 0;
    CK(cudaStreamBeginCapture(h->own_stream, cudaStreamCaptureModeThreadLocal));
    int rc = 0;
    const int G = solve_groups(h, kind, n_ep);
    if (G > 1) {
        // G episode groups on G branches of the graph: the small latency-bound kernels of one group (projection, rollouts, selection) overlap
        // the reduced-set kernel of the others, and the tail wave of one group's chains is filled by the other groups'
        cudaEventRecord(h->ev_fork, h->own_stream);
        for (int gi = 1; gi < G; gi++) cudaStreamWaitEvent(h->aux_stream[gi - 1], h->ev_fork, 0);
        for (int gi = 0; gi < G && !rc; gi++) {
            const int e0 = (int)((long long)gi * n_ep / G), e1 = (int)((long long)(gi + 1) * n_ep / G);
            int l = 0;
            const ViewSave sv = push_view(h, e0);
            rc = enqueue_solve(h, kind, e1 - e0, gi == 0 ? h->own_stream : h->aux_stream[gi - 1], &l);
            pop_view(h, sv);
            launches += l;
        }
        for (int gi = 1; gi < G; gi++) { cudaEventRecord(h->ev_join[gi - 1], h->aux_stream[gi - 1]); cudaStreamWaitEvent(h->own_stream, h->ev_join[gi - 1], 0); }
    } else rc = enqueue_solve(h, kind, n_ep, h->own_stream, &launches);
    cudaError_t ce = cudaStreamEndCapture(h->own_stream, &g);
    if (rc) { if (ce == cudaSuccess && g) cudaGraphDestroy(g); return -1; }
    CK(ce);
    if ((h->prio_mode == 1 && kind == MPCMMD_COST_MMD_OPT) || (h->prio_mode == 2 && kind != MPCMMD_COST_MMD_OPT)) {
        // Experiment (default off; measured, no effect): when the sweep's cost functions solve concurrently on one device, MPCMMD_PRIO=1 gives the kernel nodes
        // of mmd_opt graphs (the long pole) the device's highest priority, MPCMMD_PRIO=2 those of the short latency-bound cost functions.  The attribute is accepted
        // on every node, and the cvar + mmd_opt step of 25 / 50 / 100 episodes takes the same time in all three modes (profiles/r02_overlap_probe.md).
        int lo = 0, hi = 0;
        if (cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess && hi != lo) {
            size_t nn = 0; int nset = 0, nfail = 0;
            if (cudaGraphGetNodes(g, nullptr, &nn) == cudaSuccess && nn) {
                std::vector<cudaGraphNode_t> nodes(nn);
                cudaGraphGetNodes(g, nodes.data(), &nn);
                for (auto nd : nodes) {
                    cudaGraphNodeType ty;
                    if (cudaGraphNodeGetType(nd, &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
                    cudaKernelNodeAttrValue v; memset(&v, 0, sizeof(v)); v.priority = hi;
                    if (cudaGraphKernelNodeSetAttribute(nd, cudaKernelNodeAttributePriority, &v) == cudaSuccess) nset++; else nfail++;
                }
            }
            cudaGetLastError();
            if (getenv("MPCMMD_DEBUG")) fprintf(stderr, "[mpcmmd] graph kind %d n_ep %d: priority %d (range %d..%d) set on %d kernel nodes, %d failures\n", kind, n_ep, hi, lo, hi, nset, nfail);
        }
    }
    cudaGraphExec_t ge;
    ce = cudaGraphInstantiate(&ge, g, 0);
    cudaGraphDestroy(g);
    CK(ce);
    h->graphs[key] = ge;
    h->graph_launches[key] = launches;
    h->last_launches = launches;
    *out = ge;
    return 0;
}

static int check_solve_args(mpcmmd_handle_s* h, int kind, int n_ep) {
    if (!h) return fail("null handle");
    if (kind < 0 || kind > 3) return fail("mpcmmd_solve: bad cost kind");
    if (n_ep < 1 || n_ep > h->E) return fail("mpcmmd_solve: n_ep outside [1, max_episodes]");
    return 0;
}

static int solve_impl(mpcmmd_handle_s* h, int kind, int n_ep, const int32_t* idx_mpc, const float* init_state, const float* mean,
                      const float* cov, const float* x_obs, const float* y_obs, const float* v_des, const mpcmmd_out* out,
                      cudaStream_t s, cudaMemcpyKind in_kind, cudaMemcpyKind out_kind) {
    if (check_solve_args(h, kind, n_ep)) return -1;
    if (!idx_mpc || !init_state || !mean || !cov || !x_obs || !y_obs || !v_des || !out) return fail("mpcmmd_solve: null pointer");
    CK(cudaSetDevice(h->device));
    const DCfg& d = h->d; DWork& w = h->w;
    if (kind == MPCMMD_COST_MMD_OPT && ensure_opt_scratch(h)) return -1;
    cudaGraphExec_t ge;
    if (get_graph(h, kind, n_ep, &ge)) return -1;
    CK(cudaMemcpyAsync(w.idx_mpc, idx_mpc, sizeof(int32_t) * n_ep, in_kind, s));
    CK(cudaMemcpyAsync(w.init_state, init_state, sizeof(float) * 6 * n_ep, in_kind, s));
    CK(cudaMemcpyAsync(w.mean0, mean, sizeof(float) * NPAR * n_ep, in_kind, s));
    CK(cudaMemcpyAsync(w.cov0, cov, sizeof(float) * 64 * n_ep, in_kind, s));
    CK(cudaMemcpyAsync(w.x_obs, x_obs, sizeof(float) * d.O * T_ * n_ep, in_kind, s));
    CK(cudaMemcpyAsync(w.y_obs, y_obs, sizeof(float) * d.O * T_ * n_ep, in_kind, s));
    CK(cudaMemcpyAsync(w.v_des, v_des, sizeof(float) * n_ep, in_kind, s));
    CK(cudaGraphLaunch(ge, s));
    if (out->cx) CK(cudaMemcpyAsync(out->cx, w.o_cx, sizeof(float) * NV * n_ep, out_kind, s));
    if (out->cy) CK(cudaMemcpyAsync(out->cy, w.o_cy, sizeof(float) * NV * n_ep, out_kind, s));
    if (out->cost_lane) CK(cudaMemcpyAsync(out->cost_lane, w.o_lane, sizeof(float) * n_ep, out_kind, s));
    if (out->cost_obs) CK(cudaMemcpyAsync(out->cost_obs, w.o_obs, sizeof(float) * n_ep, out_kind, s));
    if (out->beta) CK(cudaMemcpyAsync(out->beta, w.o_beta, sizeof(float) * d.nr * n_ep, out_kind, s));
    if (out->sigma) CK(cudaMemcpyAsync(out->sigma, w.o_sigma, sizeof(float) * n_ep, out_kind, s));
    if (out->res_beta) CK(cudaMemcpyAsync(out->res_beta, w.o_res_beta, sizeof(float) * d.iters_in * n_ep, out_kind, s));
    return 0;
}

extern "C" int mpcmmd_solve(mpcmmd_handle h, int cost_kind, int n_ep, const int32_t* idx_mpc, const float* init_state, const float* mean,
                            const float* cov, const float* x_obs, const float* y_obs, const float* v_des, const mpcmmd_out* out, void* stream) {
    return solve_impl(h, cost_kind, n_ep, idx_mpc, init_state, mean, cov, x_obs, y_obs, v_des, out, (cudaStream_t)stream,
                      cudaMemcpyDeviceToDevice, cudaMemcpyDeviceToDevice);
}
extern "C" int mpcmmd_solve_host(mpcmmd_handle h, int cost_kind, int n_ep, const int32_t* idx_mpc, const float* init_state, const float* mean,
                                 const float* cov, const float* x_obs, const float* y_obs, const float* v_des, const mpcmmd_out* out) {
    if (!h) return fail("null handle");
    if (solve_impl(h, cost_kind, n_ep, idx_mpc, init_state, mean, cov, x_obs, y_obs, v_des, out, h->own_stream,
                   cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost)) return -1;
    CK(cudaStreamSynchronize(h->own_stream));
    return 0;
}
extern "C" int mpcmmd_last_launch_count(mpcmmd_handle h) { return h ? h->last_launches : 0; }
extern "C" const char* mpcmmd_inner_cem_path(mpcmmd_handle h) {
    if (!h) return "";
    if (!inner_cem_is_fast(h->d)) return "k_inner_cem (generic, one CTA per chain)";
    switch (h->inner_mode) {
        case INNER_WARP: return "k_inner_cem_warp (one warp per chain, persistent)";
        case INNER_CTA: return "k_inner_cem_fast (one CTA per chain)";
        case INNER_PIPE: return "k_inner_cem_pipe (two chains per CTA: 3 evaluation warps + 1 serial warp, pipelined)";
        case INNER_SPLIT: return "phase-split: k_icem_dist + 20 x (k_icem_eval + k_icem_update)";
        case INNER_CTA_LAT: return "k_inner_cem_fast<LAT> (one CTA per chain, latency build)";
        case INNER_GENERIC: return "k_inner_cem (generic, one CTA per chain)";
        default: return INNER_DEFAULT_THROUGHPUT == INNER_PIPE
                            ? "k_inner_cem_pipe (two chains per CTA: 3 evaluation warps + 1 serial warp); launches of <= 3 chains per SM: k_inner_cem_fast<LAT>"
                            : "k_inner_cem_fast (one CTA per chain); launches of <= 3 chains per SM: its latency build; <= 1 chain per SM: k_inner_cem_lat (16 warps per chain)";
    }
}

// Re-run the solve of the inputs staged by the previous mpcmmd_solve* call WITHOUT the graph, with a CUDA event after
// every launch on the launching stream, and return the device time per kernel class:
// ms[0] setup (boundary+noise+init), ms[1] projection, ms[2] rollout/risk, ms[3] select, ms[4] total; n_launch[4] likewise.
extern "C" int mpcmmd_profile_solve(mpcmmd_handle h, int cost_kind, int n_ep, float* ms, int* n_launch) {
    if (check_solve_args(h, cost_kind, n_ep)) return -1;
    if (!ms) return fail("mpcmmd_profile_solve: null pointer");
    CK(cudaSetDevice(h->device));
    std::vector<LaunchMark> marks;
    cudaEvent_t e0 = nullptr;
    cudaStream_t s = h->own_stream;
    int rc = 0;
    auto body = [&]() -> int {
        CK(cudaEventCreate(&e0));
        CK(cudaEventRecord(e0, s));
        int launches = 0;
        if (enqueue_solve(h, cost_kind, n_ep, s, &launches, &marks)) return -1;
        CK(cudaStreamSynchronize(s));
        CK(cudaGetLastError());
        for (int i = 0; i < 5; i++) { ms[i] = 0.0f; if (i < 4 && n_launch) n_launch[i] = 0; }
        cudaEvent_t prev = e0;
        for (auto& m : marks) {
            float t = 0.0f; cudaEventElapsedTime(&t, prev, m.ev);
            ms[m.cls] += t; ms[4] += t; if (n_launch) n_launch[m.cls]++;
            prev = m.ev;
        }
        return 0;
    };
    rc = body();
    if (rc) cudaStreamSynchronize(s);                    // whatever was enqueued before the failure must not outlive its events
    if (e0) cudaEventDestroy(e0);
    for (auto& m : marks) cudaEventDestroy(m.ev);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// stage entry points (synchronous, default stream)

extern "C" int mpcmmd_math_vec(int fn, const float* x, const float* y, float* out, int n, int device) {
    CK(cudaSetDevice(device));
    k_math_vec<<<(n + 255) / 256, 256>>>(fn, x, y ? y : x, out, n);
    CK(cudaDeviceSynchronize());
    return 0;
}
extern "C" int mpcmmd_rng_normal(uint32_t k0, uint32_t k1, int n, float* out, int device) {
    CK(cudaSetDevice(device));
    k_normal_table<<<(n + 255) / 256, 256>>>(k0, k1, n, out);
    CK(cudaDeviceSynchronize());
    return 0;
}
extern "C" int mpcmmd_rng_beta(uint32_t k0, uint32_t k1, const float* a, const float* b, int n, float* out, int device) {
    CK(cudaSetDevice(device));
    k_beta_table<<<(n + 127) / 128, 128>>>(k0, k1, a, b, n, out);
    CK(cudaDeviceSynchronize());
    return 0;
}
extern "C" int mpcmmd_get_tables(mpcmmd_handle h, float* z_init, float* theta0, float* zb_iter) {
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    const DCfg& d = h->d; const int dd = d.nm + 1;
    if (z_init) CK(cudaMemcpy(z_init, d.z_init, sizeof(float) * d.B * NPAR, cudaMemcpyDeviceToDevice));
    if (theta0) CK(cudaMemcpy(theta0, d.theta0, sizeof(float) * d.S_in * dd, cudaMemcpyDeviceToDevice));
    if (zb_iter) CK(cudaMemcpy(zb_iter, d.zb_iter, sizeof(float) * d.iters_in * (d.S_in - d.n_el_in) * dd, cudaMemcpyDeviceToDevice));
    return 0;
}
extern "C" int mpcmmd_stage_project(mpcmmd_handle h, int n, const float* params, const float* beq_x, const float* beq_y, float v_des,
                                    float* lam_x, float* lam_y, float* s_lane, float* cx, float* cy, float* res_norm, float* acc, float* steer,
                                    float* cost_base) {
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    float* vd = h->w.v_des;                     // one "episode": sample g -> e = g / n = 0
    CK(cudaMemcpy(vd, &v_des, sizeof(float), cudaMemcpyHostToDevice));
    ProjArgs p;
    p.n_samples = n; p.B = n; p.params = params; p.beq_x = beq_x; p.beq_y = beq_y; p.v_des = vd; p.lam_x = lam_x; p.lam_y = lam_y; p.s_lane = s_lane;
    p.cx = cx; p.cy = cy; p.res_norm = res_norm; p.cost_base = cost_base; p.acc = acc; p.steer = steer;
    { const char* dv = getenv("MPCMMD_PROJ_DEBUG"); p.dbg = dv ? atoi(dv) : 0; }
    launch_project(h, p, 0);
    CK(cudaDeviceSynchronize());
    return 0;
}
static int stage_risk_impl(mpcmmd_handle h, int cost_kind, int n, const float* acc, const float* steer, const float* state0,
                           const float* z1, const float* z2, const float* z3, const uint32_t* keys, const float* binj1, const float* binj2,
                           const float* x_obs, const float* y_obs, float* risk, float* lane, float* beta, float* sigma, float* res_beta) {
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    RiskArgs r;
    r.n_samples = n; r.B = n; r.cost_kind = cost_kind; r.acc = acc; r.steer = steer; r.state0 = state0; r.z1 = z1; r.z2 = z2; r.z3 = z3; r.z_stride = 0;
    r.keys = keys; r.key_stride = 0; r.btab = nullptr; r.btab_stride = 0; r.binj1 = binj1; r.binj2 = binj2;
    r.x_obs = x_obs; r.y_obs = y_obs; r.risk = risk; r.lane = lane; r.beta = beta; r.sigma = sigma; r.res_beta = res_beta;
    r.sx_obs = r.sy_obs = nullptr; r.obs_nan = nullptr;
    if (h->w.sx_obs) {          // many obstacles: the stage runs the product path, sorted obstacle windows included (one "episode")
        k_obs_sort<<<1, 128>>>(x_obs, y_obs, h->w.sx_obs, h->w.sy_obs, h->w.obs_nan, h->d.O, T_);
        r.sx_obs = h->w.sx_obs; r.sy_obs = h->w.sy_obs; r.obs_nan = h->w.obs_nan;
    }
    if (cost_kind == MPCMMD_COST_MMD_OPT && ensure_opt_scratch(h)) return -1;
    if (launch_risk(h, r, 0)) return -1;
    CK(cudaDeviceSynchronize());
    return 0;
}
extern "C" int mpcmmd_stage_risk(mpcmmd_handle h, int cost_kind, int n, const float* acc, const float* steer, const float* state0,
                                 const float* z1, const float* z2, const float* z3, const uint32_t* keys, const float* x_obs, const float* y_obs,
                                 float* risk, float* lane, float* beta, float* sigma, float* res_beta) {
    return stage_risk_impl(h, cost_kind, n, acc, steer, state0, z1, z2, z3, keys, nullptr, nullptr, x_obs, y_obs, risk, lane, beta, sigma, res_beta);
}
// the same stage with the random draws of the beta noise model INJECTED: beta_acc / beta_steer (n, nr*np) are the samples of
// jax.random.beta(key, 2|u|, 5|u|) at cem_helper.py:427 / :432 (:492 / :497), z3 (nr*np) the common-mode normals.  No device RNG runs.
extern "C" int mpcmmd_stage_risk_injected(mpcmmd_handle h, int cost_kind, int n, const float* acc, const float* steer, const float* state0,
                                          const float* z3, const float* beta_acc, const float* beta_steer, const float* x_obs, const float* y_obs,
                                          float* risk, float* lane, float* beta, float* sigma, float* res_beta) {
    if (!h) return fail("null handle");
    if (h->d.noise_kind != 1) return fail("mpcmmd_stage_risk_injected: the handle was not created with beta noise (gaussian draws are injected through mpcmmd_stage_risk's z1, z2, z3)");
    if (!beta_acc || !beta_steer || !z3) return fail("mpcmmd_stage_risk_injected: null draw tensor");
    return stage_risk_impl(h, cost_kind, n, acc, steer, state0, z3, z3, z3, (const uint32_t*)h->w.keys, beta_acc, beta_steer, x_obs, y_obs, risk, lane, beta, sigma, res_beta);
}
extern "C" int mpcmmd_stage_select(mpcmmd_handle h, int cost_kind, const float* res_norm, const float* risk, const float* cost_base, float* params,
                                   float* mean, float* cov, const float* z_cem, int32_t* sel) {
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    const DCfg& d = h->d; DWork& w = h->w;
    SelArgs a;
    a.n_ep = 1; a.B = d.B; a.it = 0; a.nr = d.nr; a.iters_in = d.iters_in; a.w_obs = w_obs_for(h, cost_kind);
    a.res_norm = res_norm; a.risk = risk; a.lane = w.lane; a.cost_base = cost_base; a.params = params; a.mean = mean; a.cov = cov;
    a.zcem = z_cem; a.z_stride = 0; a.cx = w.cx; a.cy = w.cy; a.beta = w.beta; a.sigma = w.sigma; a.res_beta = w.res_beta;
    a.o_cx = w.o_cx; a.o_cy = w.o_cy; a.o_lane = w.o_lane; a.o_obs = w.o_obs; a.o_beta = w.o_beta; a.o_sigma = w.o_sigma; a.o_res_beta = w.o_res_beta;
    a.o_sel = sel; a.sel_stride = 1;
    k_select<<<1, d.B <= SEL_RANK_MAX ? SEL_THREADS : SEL_THREADS_BIG, sel_smem(d)>>>(d, a);
    CK(cudaDeviceSynchronize());
    return 0;
}
// the initial CEM batch of one episode (Helper.sampling_param, cem_helper.py:122-150): k_init on (mean, cov), all DEVICE pointers
extern "C" int mpcmmd_stage_init(mpcmmd_handle h, const float* mean, const float* cov, float* params) {
    if (!h) return fail("null handle");
    if (!mean || !cov || !params) return fail("mpcmmd_stage_init: null pointer");
    CK(cudaSetDevice(h->device));
    const DCfg& d = h->d; DWork& w = h->w;
    CK(cudaMemcpy(w.mean0, mean, sizeof(float) * NPAR, cudaMemcpyDeviceToDevice));
    CK(cudaMemcpy(w.cov0, cov, sizeof(float) * 64, cudaMemcpyDeviceToDevice));
    k_init<<<1, d.B <= SEL_RANK_MAX ? 128 : 1024>>>(d, w, 1);
    CK(cudaDeviceSynchronize());
    CK(cudaMemcpy(params, w.params, sizeof(float) * d.B * NPAR, cudaMemcpyDeviceToDevice));
    return 0;
}
extern "C" int mpcmmd_stage_noise(mpcmmd_handle h, int32_t idx_mpc, int32_t iter, float* z1, float* z2, float* z3, float* z_cem, uint32_t* keys) {
    if (!h) return fail("null handle");
    CK(cudaSetDevice(h->device));
    const DCfg& d = h->d; DWork& w = h->w;
    if (iter < 0 || iter >= d.iters) return fail("mpcmmd_stage_noise: iter outside [0, maxiter_cem)");
    const size_t n = (size_t)d.nr * d.np, ncem = (size_t)(d.B - d.n_el) * NPAR;
    CK(cudaMemcpy(w.idx_mpc, &idx_mpc, sizeof(int32_t), cudaMemcpyHostToDevice));
    DCfg dg = d; dg.noise_kind = 0;                                  // always emit the Gaussian tables here
    k_noise<<<1, 128>>>(dg, w, 1, iter, 1);
    CK(cudaDeviceSynchronize());
    const size_t slot = (size_t)iter;
    if (z1) CK(cudaMemcpy(z1, w.z1 + slot * n, sizeof(float) * n, cudaMemcpyDeviceToDevice));
    if (z2) CK(cudaMemcpy(z2, w.z2 + slot * n, sizeof(float) * n, cudaMemcpyDeviceToDevice));
    if (z3) CK(cudaMemcpy(z3, w.z3 + slot * n, sizeof(float) * n, cudaMemcpyDeviceToDevice));
    if (z_cem) CK(cudaMemcpy(z_cem, w.zcem + slot * ncem, sizeof(float) * ncem, cudaMemcpyDeviceToDevice));
    if (keys) CK(cudaMemcpy(keys, w.keys + slot * 4, sizeof(uint32_t) * 4, cudaMemcpyDeviceToDevice));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Monte-Carlo validation (S/validation.py:134-171): host arrays in, counts out.  Not tied to a handle.
// k_validate on device arrays: the rollout + counting half shared by both validation entry points (enqueue only).
static cudaError_t launch_validate(int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, double dt, double wheel_base, double a_obs,
                                   double b_obs, double y_lb, double y_ub, size_t smem, const double* d_acc, const double* d_steer,
                                   const double* d_s0, const double* d_xo, const double* d_yo, int32_t* d_cnt, int32_t* d_lane,
                                   double* d_xr, double* d_yr) {
    if (smem > 48 * 1024) {
        const cudaError_t e = cudaFuncSetAttribute(k_validate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    ValCfg c;
    c.n_roll = n_roll; c.np = num_prime; c.O = num_obs; c.obs_f32 = obs_cost_f32; c.dt = dt; c.wheel_base = wheel_base;
    c.a2 = a_obs * a_obs; c.b2 = b_obs * b_obs; c.y_lb = y_lb; c.y_ub = y_ub;
    k_validate<<<n_ep, VAL_THREADS, smem>>>(c, d_acc, d_steer, d_s0, d_xo, d_yo, d_cnt, d_lane, d_xr, d_yr);
    return cudaGetLastError();
}

extern "C" int mpcmmd_validate_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, double dt, double wheel_base,
                                    double a_obs, double b_obs, double y_lb, double y_ub, const double* acc, const double* steer,
                                    const double* state0, const double* x_obs_traj, const double* y_obs_traj, int32_t* count,
                                    int32_t* count_lane, double* x_roll, double* y_roll) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("mpcmmd_validate_host: no CUDA device (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail("mpcmmd_validate_host: bad device index");
    if (n_ep < 1 || n_roll < 1 || num_prime < 1 || num_prime > MPCMMD_T || num_obs < 1) return fail("mpcmmd_validate_host: bad sizes");
    if (!acc || !steer || !state0 || !x_obs_traj || !y_obs_traj || !count || !count_lane) return fail("mpcmmd_validate_host: null pointer");
    if ((x_roll == nullptr) != (y_roll == nullptr)) return fail("mpcmmd_validate_host: x_roll and y_roll must both be given or both be null");
    const size_t smem = (size_t)(num_obs + 2) * num_prime * sizeof(int);
    if (smem > 200 * 1024) return fail("mpcmmd_validate_host: (num_obs + 2) * num_prime counters do not fit in shared memory");
    CK(cudaSetDevice(device));
    const size_t nc = (size_t)n_ep * n_roll * num_prime, no = (size_t)n_ep * num_obs * num_prime;
    double *d_acc = nullptr, *d_steer = nullptr, *d_s0 = nullptr, *d_xo = nullptr, *d_yo = nullptr, *d_xr = nullptr, *d_yr = nullptr;
    int32_t *d_cnt = nullptr, *d_lane = nullptr;
    int rc = 0;
    auto body = [&]() -> int {
        CK(cudaMalloc(&d_acc, nc * 8)); CK(cudaMalloc(&d_steer, nc * 8)); CK(cudaMalloc(&d_s0, (size_t)n_ep * 5 * 8));
        CK(cudaMalloc(&d_xo, no * 8)); CK(cudaMalloc(&d_yo, no * 8)); CK(cudaMalloc(&d_cnt, (size_t)n_ep * 4)); CK(cudaMalloc(&d_lane, (size_t)n_ep * 4));
        if (x_roll) { CK(cudaMalloc(&d_xr, nc * 8)); CK(cudaMalloc(&d_yr, nc * 8)); }
        CK(cudaMemcpy(d_acc, acc, nc * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_steer, steer, nc * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_s0, state0, (size_t)n_ep * 5 * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_xo, x_obs_traj, no * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_yo, y_obs_traj, no * 8, cudaMemcpyHostToDevice));
        CK(launch_validate(n_ep, n_roll, num_prime, num_obs, obs_cost_f32, dt, wheel_base, a_obs, b_obs, y_lb, y_ub, smem,
                           d_acc, d_steer, d_s0, d_xo, d_yo, d_cnt, d_lane, d_xr, d_yr));
        CK(cudaMemcpy(count, d_cnt, (size_t)n_ep * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(count_lane, d_lane, (size_t)n_ep * 4, cudaMemcpyDeviceToHost));
        if (x_roll) { CK(cudaMemcpy(x_roll, d_xr, nc * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(y_roll, d_yr, nc * 8, cudaMemcpyDeviceToHost)); }
        return 0;
    };
    rc = body();
    cudaFree(d_acc); cudaFree(d_steer); cudaFree(d_s0); cudaFree(d_xo); cudaFree(d_yo); cudaFree(d_cnt); cudaFree(d_lane); cudaFree(d_xr); cudaFree(d_yr);
    return rc;
}

// The same with the noise drawn on the device (k_validate_noise): planned controls and per-trajectory seeds in, counts out.
extern "C" int mpcmmd_validate_seeded_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, int noise_kind,
                                           double noise_level, double k_steer, double beta_a, double beta_b, double acc_const_noise,
                                           double steer_const_noise, double dt, double wheel_base, double a_obs, double b_obs, double y_lb,
                                           double y_ub, const uint32_t* seed, const double* acc_plan, const double* steer_plan,
                                           const double* state0, const double* x_obs_traj, const double* y_obs_traj, int32_t* count,
                                           int32_t* count_lane, double* acc_out, double* steer_out, uint32_t* state_out) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("mpcmmd_validate_seeded_host: no CUDA device (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail("mpcmmd_validate_seeded_host: bad device index");
    if (n_ep < 1 || n_roll < 1 || num_prime < 1 || num_prime > MPCMMD_T || num_obs < 1) return fail("mpcmmd_validate_seeded_host: bad sizes");
    if (noise_kind != 0 && noise_kind != 1) return fail("mpcmmd_validate_seeded_host: noise_kind must be 0 (gaussian) or 1 (beta)");
    if (!seed || !acc_plan || !steer_plan || !state0 || !x_obs_traj || !y_obs_traj || !count || !count_lane)
        return fail("mpcmmd_validate_seeded_host: null pointer");
    if ((acc_out == nullptr) != (steer_out == nullptr)) return fail("mpcmmd_validate_seeded_host: acc_out and steer_out must both be given or both be null");
    if (noise_kind == 1) {                               // np.random.beta's argument check (NaN passes), before anything is drawn
        for (size_t i = 0; i < (size_t)n_ep * num_prime; i++) {
            if (beta_a * fabs(acc_plan[i]) <= 0.0 || beta_a * fabs(steer_plan[i]) + 1e-5 <= 0.0) return fail("mpcmmd_validate_seeded_host: a <= 0");
            if (beta_b * fabs(acc_plan[i]) <= 0.0 || beta_b * fabs(steer_plan[i]) + 1e-5 <= 0.0) return fail("mpcmmd_validate_seeded_host: b <= 0");
        }
    }
    const size_t smem = (size_t)(num_obs + 2) * num_prime * sizeof(int);
    if (smem > 200 * 1024) return fail("mpcmmd_validate_seeded_host: (num_obs + 2) * num_prime counters do not fit in shared memory");
    CK(cudaSetDevice(device));
    const size_t nc = (size_t)n_ep * n_roll * num_prime, no = (size_t)n_ep * num_obs * num_prime, npl = (size_t)n_ep * num_prime;
    double *d_ap = nullptr, *d_sp = nullptr, *d_acc = nullptr, *d_steer = nullptr, *d_s0 = nullptr, *d_xo = nullptr, *d_yo = nullptr;
    uint32_t *d_seed = nullptr, *d_state = nullptr;
    int32_t *d_cnt = nullptr, *d_lane = nullptr;
    auto body = [&]() -> int {
        CK(cudaMalloc(&d_seed, (size_t)n_ep * 4)); CK(cudaMalloc(&d_ap, npl * 8)); CK(cudaMalloc(&d_sp, npl * 8));
        CK(cudaMalloc(&d_acc, nc * 8)); CK(cudaMalloc(&d_steer, nc * 8)); CK(cudaMalloc(&d_s0, (size_t)n_ep * 5 * 8));
        CK(cudaMalloc(&d_xo, no * 8)); CK(cudaMalloc(&d_yo, no * 8)); CK(cudaMalloc(&d_cnt, (size_t)n_ep * 4)); CK(cudaMalloc(&d_lane, (size_t)n_ep * 4));
        if (state_out) CK(cudaMalloc(&d_state, (size_t)n_ep * VALN_STATE_WORDS * 4));
        CK(cudaMemcpy(d_seed, seed, (size_t)n_ep * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_ap, acc_plan, npl * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_sp, steer_plan, npl * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_s0, state0, (size_t)n_ep * 5 * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_xo, x_obs_traj, no * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_yo, y_obs_traj, no * 8, cudaMemcpyHostToDevice));
        ValNoiseCfg vn;
        vn.n_roll = n_roll; vn.np = num_prime; vn.noise_kind = noise_kind; vn.nl = noise_level; vn.k_steer = k_steer;
        vn.beta_a = beta_a; vn.beta_b = beta_b; vn.c_acc = acc_const_noise; vn.c_steer = steer_const_noise;
        k_validate_noise<<<n_ep, VALN_THREADS>>>(vn, d_seed, d_ap, d_sp, d_acc, d_steer, d_state);
        CK(cudaGetLastError());
        CK(launch_validate(n_ep, n_roll, num_prime, num_obs, obs_cost_f32, dt, wheel_base, a_obs, b_obs, y_lb, y_ub, smem,
                           d_acc, d_steer, d_s0, d_xo, d_yo, d_cnt, d_lane, nullptr, nullptr));
        CK(cudaMemcpy(count, d_cnt, (size_t)n_ep * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(count_lane, d_lane, (size_t)n_ep * 4, cudaMemcpyDeviceToHost));
        if (acc_out) { CK(cudaMemcpy(acc_out, d_acc, nc * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(steer_out, d_steer, nc * 8, cudaMemcpyDeviceToHost)); }
        if (state_out) CK(cudaMemcpy(state_out, d_state, (size_t)n_ep * VALN_STATE_WORDS * 4, cudaMemcpyDeviceToHost));
        return 0;
    };
    const int rc = body();
    cudaFree(d_seed); cudaFree(d_ap); cudaFree(d_sp); cudaFree(d_acc); cudaFree(d_steer); cudaFree(d_s0); cudaFree(d_xo); cudaFree(d_yo);
    cudaFree(d_cnt); cudaFree(d_lane); cudaFree(d_state);
    return rc;
}

// The same with counter-based noise (k_validate_jax, DESIGN.md section 3 item 7): each rollout draws its JAX-protocol noise while it
// rolls out, so n_roll is bounded only by JAX's uint32 element counters.
extern "C" int mpcmmd_validate_threefry_host(int device, int n_ep, int n_roll, int num_prime, int num_obs, int obs_cost_f32, int noise_kind,
                                             double noise_level, double k_steer, double beta_a, double beta_b, double acc_const_noise,
                                             double steer_const_noise, double dt, double wheel_base, double a_obs, double b_obs, double y_lb,
                                             double y_ub, const uint32_t* seed, const double* acc_plan, const double* steer_plan,
                                             const double* state0, const double* x_obs_traj, const double* y_obs_traj, int32_t* count,
                                             int32_t* count_lane, double* acc_out, double* steer_out) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return fail("mpcmmd_validate_threefry_host: no CUDA device (this library has no CPU fallback)");
    if (device < 0 || device >= ndev) return fail("mpcmmd_validate_threefry_host: bad device index");
    if (n_roll < 1) return fail("mpcmmd_validate_threefry_host: n_roll must be >= 1");
    if (n_ep < 1 || num_prime < 1 || num_prime > MPCMMD_T || num_obs < 1) return fail("mpcmmd_validate_threefry_host: bad sizes");
    if ((long long)n_roll * num_prime >= (1LL << 31))
        return fail("mpcmmd_validate_threefry_host: n_roll * num_prime must be below 2^31 (JAX's uint32 element counters)");
    if (noise_kind != 0 && noise_kind != 1) return fail("mpcmmd_validate_threefry_host: noise_kind must be 0 (gaussian) or 1 (beta)");
    if (!seed || !acc_plan || !steer_plan || !state0 || !x_obs_traj || !y_obs_traj || !count || !count_lane)
        return fail("mpcmmd_validate_threefry_host: null pointer");
    if ((acc_out == nullptr) != (steer_out == nullptr)) return fail("mpcmmd_validate_threefry_host: acc_out and steer_out must both be given or both be null");
    const size_t smem = (size_t)(num_obs + 2) * num_prime * sizeof(int);
    if (smem > 200 * 1024) return fail("mpcmmd_validate_threefry_host: (num_obs + 2) * num_prime counters do not fit in shared memory");
    CK(cudaSetDevice(device));
    const size_t nc = (size_t)n_ep * n_roll * num_prime, no = (size_t)n_ep * num_obs * num_prime, npl = (size_t)n_ep * num_prime;
    const size_t ncnt = (size_t)n_ep * (num_obs + 2) * num_prime;
    double *d_ap = nullptr, *d_sp = nullptr, *d_acc = nullptr, *d_steer = nullptr, *d_s0 = nullptr, *d_xo = nullptr, *d_yo = nullptr;
    uint32_t* d_seed = nullptr;
    int32_t *d_cg = nullptr, *d_cnt = nullptr, *d_lane = nullptr;
    auto body = [&]() -> int {
        CK(cudaMalloc(&d_seed, (size_t)n_ep * 4)); CK(cudaMalloc(&d_ap, npl * 8)); CK(cudaMalloc(&d_sp, npl * 8));
        CK(cudaMalloc(&d_s0, (size_t)n_ep * 5 * 8)); CK(cudaMalloc(&d_xo, no * 8)); CK(cudaMalloc(&d_yo, no * 8));
        CK(cudaMalloc(&d_cg, ncnt * 4)); CK(cudaMalloc(&d_cnt, (size_t)n_ep * 4)); CK(cudaMalloc(&d_lane, (size_t)n_ep * 4));
        if (acc_out) { CK(cudaMalloc(&d_acc, nc * 8)); CK(cudaMalloc(&d_steer, nc * 8)); }
        CK(cudaMemcpy(d_seed, seed, (size_t)n_ep * 4, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_ap, acc_plan, npl * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_sp, steer_plan, npl * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_s0, state0, (size_t)n_ep * 5 * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(d_xo, x_obs_traj, no * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(d_yo, y_obs_traj, no * 8, cudaMemcpyHostToDevice));
        CK(cudaMemset(d_cg, 0, ncnt * 4));
        if (smem > 48 * 1024) CK(cudaFuncSetAttribute(k_validate_jax, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ValCfg c;
        c.n_roll = n_roll; c.np = num_prime; c.O = num_obs; c.obs_f32 = obs_cost_f32; c.dt = dt; c.wheel_base = wheel_base;
        c.a2 = a_obs * a_obs; c.b2 = b_obs * b_obs; c.y_lb = y_lb; c.y_ub = y_ub;
        ValJaxCfg j;
        j.noise_kind = noise_kind; j.nl = noise_level; j.ks = k_steer * noise_level; j.beta_a = beta_a; j.beta_b = beta_b;
        j.c_acc = acc_const_noise; j.c_steer = steer_const_noise;
        const unsigned chunks = (unsigned)((n_roll + VALJ_THREADS - 1) / VALJ_THREADS);
        for (int e0 = 0; e0 < n_ep; e0 += 65535) {                      // gridDim.y <= 65535 trajectories per launch
            const dim3 grid(chunks, (unsigned)(n_ep - e0 < 65535 ? n_ep - e0 : 65535));
            k_validate_jax<<<grid, VALJ_THREADS, smem>>>(c, j, e0, d_seed, d_ap, d_sp, d_s0, d_xo, d_yo, d_cg, d_acc, d_steer);
            CK(cudaGetLastError());
        }
        k_validate_finish<<<n_ep, 32>>>(num_obs, num_prime, d_cg, d_cnt, d_lane);
        CK(cudaGetLastError());
        CK(cudaMemcpy(count, d_cnt, (size_t)n_ep * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(count_lane, d_lane, (size_t)n_ep * 4, cudaMemcpyDeviceToHost));
        if (acc_out) { CK(cudaMemcpy(acc_out, d_acc, nc * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(steer_out, d_steer, nc * 8, cudaMemcpyDeviceToHost)); }
        return 0;
    };
    const int rc = body();
    cudaFree(d_seed); cudaFree(d_ap); cudaFree(d_sp); cudaFree(d_acc); cudaFree(d_steer); cudaFree(d_s0); cudaFree(d_xo); cudaFree(d_yo);
    cudaFree(d_cg); cudaFree(d_cnt); cudaFree(d_lane);
    return rc;
}

// ------------------------------------------------------------------------------------------------
// FP32 FMA peak of this device, measured (the roofline denominator for the FP32-bound kernels; MEASURED_PEAKS.json
// has only HBM and bf16-GEMM peaks).  8 independent fma chains per thread, 2048 threads per SM resident.
__global__ void __launch_bounds__(256) k_fma_peak(float* out, int iters, float a, float b) {
    float x0 = threadIdx.x * 1e-3f, x1 = x0 + 1.0f, x2 = x0 + 2.0f, x3 = x0 + 3.0f, x4 = x0 + 4.0f, x5 = x0 + 5.0f, x6 = x0 + 6.0f, x7 = x0 + 7.0f;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 16; u++) {
            x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
            x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}
extern "C" int mpcmmd_fp32_peak(int device, float* tflops, int* sm_count) {
    CK(cudaSetDevice(device));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 4096;
    float* buf; CK(cudaMalloc(&buf, sizeof(float) * blocks * threads));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    float best = 0.0f;
    for (int rep = 0; rep < 6; rep++) {
        CK(cudaEventRecord(e0));
        k_fma_peak<<<blocks, threads>>>(buf, iters, 0.999f, 1e-3f);
        CK(cudaEventRecord(e1));
        CK(cudaEventSynchronize(e1));
        float ms = 0.0f; CK(cudaEventElapsedTime(&ms, e0, e1));
        const double flop = 2.0 * 8 * 16 * (double)iters * blocks * threads;
        const float tf = (float)(flop / (ms * 1e-3) / 1e12);
        if (rep > 0 && tf > best) best = tf;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf);
    *tflops = best;
    if (sm_count) *sm_count = prop.multiProcessorCount;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// XU / special-function peaks of this device, measured (SURVEY.md section 8d asks for an `ex2` peak next to the FP32-FMA one): the denominators
// for the kernels whose hot instructions are MUFU (ex2.approx) or the IEEE division / square root sequences (MUFU.RCP / MUFU.RSQ + Newton
// steps on the FMA pipe) -- k_rollouts' obstacle indicator divides twice per (point, obstacle), the bicycle step takes one sqrt.
// out[0] = ex2.approx.ftz.f32 Gop/s, out[1] = div.rn.f32 Gop/s, out[2] = sqrt.rn.f32 Gop/s (thread-level operations per second / 1e9).
template <int OP>
__global__ void __launch_bounds__(256) k_xu_peak(float* out, int iters, float a) {
    float x0 = 0.5f + threadIdx.x * 1e-4f, x1 = x0 + 0.01f, x2 = x0 + 0.02f, x3 = x0 + 0.03f, x4 = x0 + 0.04f, x5 = x0 + 0.05f, x6 = x0 + 0.06f, x7 = x0 + 0.07f;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            if (OP == 0) {
#define XU_EX2(v) asm volatile("ex2.approx.ftz.f32 %0, %1;" : "=f"(v) : "f"(-v))
                XU_EX2(x0); XU_EX2(x1); XU_EX2(x2); XU_EX2(x3); XU_EX2(x4); XU_EX2(x5); XU_EX2(x6); XU_EX2(x7);
#undef XU_EX2
            } else if (OP == 1) {
                x0 = __fdiv_rn(a, x0); x1 = __fdiv_rn(a, x1); x2 = __fdiv_rn(a, x2); x3 = __fdiv_rn(a, x3);
                x4 = __fdiv_rn(a, x4); x5 = __fdiv_rn(a, x5); x6 = __fdiv_rn(a, x6); x7 = __fdiv_rn(a, x7);
            } else {
                x0 = __fsqrt_rn(x0 + a); x1 = __fsqrt_rn(x1 + a); x2 = __fsqrt_rn(x2 + a); x3 = __fsqrt_rn(x3 + a);
                x4 = __fsqrt_rn(x4 + a); x5 = __fsqrt_rn(x5 + a); x6 = __fsqrt_rn(x6 + a); x7 = __fsqrt_rn(x7 + a);
            }
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
}
// ---- exhaustive check of the IEEE shortcuts of dmath.cuh (dm::sqrt_rcp, dm::div10) against sqrtf / the IEEE division on every float bit pattern
__global__ void k_selfcheck_ieee(unsigned long long* bad /* [3] */) {
    unsigned long long b0 = 0, b1 = 0, b2 = 0;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < (1ULL << 32); i += stride) {
        const float a = dm::u2f((uint32_t)i);
        float dd, rd; dm::sqrt_rcp(a, dd, rd);
        const float ds = sqrtf(a), rs = 1.0f / ds;
        b0 += !(dm::f2u(dd) == dm::f2u(ds) || (dd != dd && ds != ds));
        b1 += !(dm::f2u(rd) == dm::f2u(rs) || (rd != rd && rs != rs));
        const float q = dm::div10(a), qs = a / 10.0f;
        b2 += !(dm::f2u(q) == dm::f2u(qs) || (q != q && qs != qs));
    }
    if (b0) atomicAdd(bad, b0);
    if (b1) atomicAdd(bad + 1, b1);
    if (b2) atomicAdd(bad + 2, b2);
}
extern "C" int mpcmmd_selfcheck_ieee(int device, unsigned long long* mismatches /* [3], host */) {
    if (!mismatches) return fail("mpcmmd_selfcheck_ieee: null pointer");
    CK(cudaSetDevice(device));
    unsigned long long* d = nullptr;
    CK(cudaMalloc(&d, 3 * sizeof(unsigned long long)));
    cudaMemset(d, 0, 3 * sizeof(unsigned long long));
    k_selfcheck_ieee<<<148 * 8, 256>>>(d);
    cudaError_t e = cudaDeviceSynchronize();
    if (e == cudaSuccess) e = cudaMemcpy(mismatches, d, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    cudaFree(d);
    CK(e);
    return 0;
}

extern "C" int mpcmmd_xu_peaks(int device, float* gops /* [3] */) {
    if (!gops) return fail("mpcmmd_xu_peaks: null pointer");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device));
    const int blocks = prop.multiProcessorCount * 8, threads = 256, iters = 512;
    float* buf; CK(cudaMalloc(&buf, sizeof(float) * blocks * threads));
    cudaEvent_t e0, e1; CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    for (int op = 0; op < 3; op++) {
        float best = 0.0f;
        for (int rep = 0; rep < 5; rep++) {
            CK(cudaEventRecord(e0));
            if (op == 0) k_xu_peak<0><<<blocks, threads>>>(buf, iters, 1.25f);
            else if (op == 1) k_xu_peak<1><<<blocks, threads>>>(buf, iters, 1.25f);
            else k_xu_peak<2><<<blocks, threads>>>(buf, iters, 1.25f);
            CK(cudaEventRecord(e1));
            CK(cudaEventSynchronize(e1));
            float ms = 0.0f; CK(cudaEventElapsedTime(&ms, e0, e1));
            const double ops = 8.0 * 8 * (double)iters * blocks * threads;
            const float g = (float)(ops / (ms * 1e-3) / 1e9);
            if (rep > 0 && g > best) best = g;
        }
        gops[op] = best;
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(buf);
    return 0;
}
