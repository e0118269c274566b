/* oracle_nprng.h -- plain-C restatement of NumPy's legacy RandomState stream as the reference's validation.py consumes it
 * (np.random.seed(key); beta / multivariate_normal, validation.py:43-84).  TEST INFRASTRUCTURE ONLY.
 *
 * The contract is DESIGN.md section 3 item 6 (the "NumPy legacy stream").  NumPy's legacy generator is frozen (NEP 19); the functions
 * below follow numpy/random/src/mt19937 (seed, twist, next32, next_double) and numpy/random/src/legacy/legacy-distributions.c
 * (legacy_gauss, legacy_standard_exponential, legacy_standard_gamma, legacy_beta) one for one.  pow / log / exp / sqrt are the C
 * library's, as in NumPy, so built with -ffp-contract=off against glibc this reproduces NumPy bit for bit.
 * csrc/dnprng.cuh is the device mirror, function for function. */
#pragma once
#include <math.h>
#include <stdint.h>

#define NPR_N 624
#define NPR_M 397

typedef struct {
    uint32_t key[NPR_N];
    int pos, has_gauss;
    double gauss;
} npr_state;

/* np.random.seed(k) with a Python int in [0, 2^32 - 1]: init_genrand */
static void npr_seed(npr_state *s, uint32_t seed) {
    for (int i = 0; i < NPR_N; i++) {
        s->key[i] = seed;
        seed = 1812433253u * (seed ^ (seed >> 30)) + (uint32_t)(i + 1);
    }
    s->pos = NPR_N; s->has_gauss = 0; s->gauss = 0.0;
}

static void npr_twist(npr_state *s) {
    uint32_t *k = s->key;
    for (int i = 0; i < NPR_N; i++) {
        const uint32_t y = (k[i] & 0x80000000u) | (k[(i + 1) % NPR_N] & 0x7fffffffu);
        k[i] = k[(i + NPR_M) % NPR_N] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    s->pos = 0;
}

static uint32_t npr_u32(npr_state *s) {
    if (s->pos == NPR_N) npr_twist(s);
    uint32_t y = s->key[s->pos++];
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    return y;
}

/* 53-bit double in [0, 1): the first word gives the high 27 bits */
static double npr_double(npr_state *s) {
    const int32_t a = (int32_t)(npr_u32(s) >> 5);
    const int32_t b = (int32_t)(npr_u32(s) >> 6);
    return (a * 67108864.0 + b) / 9007199254740992.0;
}

/* polar method with a one-value cache; consuming the cache zeroes it (get_state() shows gauss = 0.0 then) */
static double npr_gauss(npr_state *s) {
    if (s->has_gauss) {
        const double t = s->gauss;
        s->has_gauss = 0; s->gauss = 0.0;
        return t;
    }
    double x1, x2, r2;
    do {
        x1 = 2.0 * npr_double(s) - 1.0;
        x2 = 2.0 * npr_double(s) - 1.0;
        r2 = x1 * x1 + x2 * x2;
    } while (r2 >= 1.0 || r2 == 0.0);
    const double f = sqrt(-2.0 * log(r2) / r2);
    s->gauss = f * x1; s->has_gauss = 1;
    return f * x2;
}

static double npr_exponential(npr_state *s) { return -log(1.0 - npr_double(s)); }

static double npr_gamma(npr_state *s, double shape) {
    if (shape == 1.0) return npr_exponential(s);
    if (shape == 0.0) return 0.0;
    if (shape < 1.0) {
        for (;;) {
            const double U = npr_double(s), V = npr_exponential(s);
            if (U <= 1.0 - shape) {
                const double X = pow(U, 1. / shape);
                if (X <= V) return X;
            } else {
                const double Y = -log((1 - U) / shape);
                const double X = pow(1.0 - shape + shape * Y, 1. / shape);
                if (X <= (V + Y)) return X;
            }
        }
    }
    const double b = shape - 1. / 3., c = 1. / sqrt(9 * b);
    for (;;) {
        double X, V;
        do {
            X = npr_gauss(s);
            V = 1.0 + c * X;
        } while (V <= 0.0);
        V = V * V * V;
        const double U = npr_double(s);
        if (U < 1.0 - 0.0331 * (X * X) * (X * X)) return b * V;
        if (log(U) < 0.5 * X * X + b * (1. - V + log(V))) return b * V;
    }
}

static double npr_beta(npr_state *s, double a, double b) {
    if (a <= 1.0 && b <= 1.0) {                                 /* Johnk */
        for (;;) {
            const double U = npr_double(s), V = npr_double(s);
            const double X = pow(U, 1.0 / a), Y = pow(V, 1.0 / b);
            if ((X + Y) <= 1.0) {
                if (X + Y > 0) return X / (X + Y);
                double lx = log(U) / a, ly = log(V) / b;    /* both powers underflowed: log space */
                const double lm = lx > ly ? lx : ly;
                lx -= lm; ly -= lm;
                return exp(lx - log(exp(lx) + exp(ly)));
            }
        }
    }
    const double Ga = npr_gamma(s, a), Gb = npr_gamma(s, b);
    return Ga / (Ga + Gb);
}

/* The noisy controls of one trajectory (validation.py:40-90 = mpcmmd_b200.validation.perturbed_controls) from a freshly seeded
 * stream: noise_kind 1 (beta) draws beta(a|acc|, b|acc|, (n_roll, np)), beta(a|steer| + 1e-5, b|steer| + 1e-5, (n_roll, np)), then
 * multivariate_normal(0, I, (n_roll,)); noise_kind 0 (gaussian) three multivariate_normal(0, I, (n_roll,)).  multivariate_normal(0, I)
 * is standard_normal in row-major order plus the mean 0.0.  acc_out, steer_out (n_roll, np), float64 with the reference's association:
 * (plan + perturbation) + c * z. */
static void npr_perturbed(npr_state *s, int noise_kind, int n_roll, int np, const double *acc, const double *steer, double nl, double k_steer,
                          double beta_a, double beta_b, double c_acc, double c_steer, double *acc_out, double *steer_out) {
    if (noise_kind == 1) {
        for (int r = 0; r < n_roll; r++)
            for (int t = 0; t < np; t++)
                acc_out[r * np + t] = acc[t] + nl * (2 * npr_beta(s, beta_a * fabs(acc[t]), beta_b * fabs(acc[t])) - 1);
        for (int r = 0; r < n_roll; r++)
            for (int t = 0; t < np; t++)
                steer_out[r * np + t] = steer[t] + (k_steer * nl) * (2 * npr_beta(s, beta_a * fabs(steer[t]) + 1e-5, beta_b * fabs(steer[t]) + 1e-5) - 1);
    } else {
        for (int r = 0; r < n_roll; r++)
            for (int t = 0; t < np; t++)
                acc_out[r * np + t] = acc[t] + (nl * fabs(acc[t])) * (npr_gauss(s) + 0.0);
        for (int r = 0; r < n_roll; r++)
            for (int t = 0; t < np; t++)
                steer_out[r * np + t] = steer[t] + (nl * fabs(steer[t])) * (npr_gauss(s) + 0.0);
    }
    for (int r = 0; r < n_roll; r++)
        for (int t = 0; t < np; t++) {
            const double z = npr_gauss(s) + 0.0;
            acc_out[r * np + t] = acc_out[r * np + t] + c_acc * z;
            steer_out[r * np + t] = steer_out[r * np + t] + c_steer * z;
        }
}
