// dnprng.cuh -- device restatement of NumPy's legacy RandomState stream as the reference's validation.py consumes it
// (np.random.seed(key); beta / multivariate_normal, S/validation.py:43-84).  Mirror of tests/nprng/oracle_nprng.h function for
// function (the contract: DESIGN.md section 3 item 6).  Stream consumption is exact: every u32 is the one NumPy draws, every
// rejection test is NumPy's.  The values differ from NumPy's only where CUDA's double pow / log / exp round differently from
// glibc's (sqrt and / are IEEE on both sides); no intrinsics, no fast math, and --fmad=false keeps the reference's association.
// One deliberate difference in form: pow goes through pow_np, which repairs CUDA's pow in the subnormal range.
#pragma once
#include <stdint.h>

namespace dnp {

constexpr int N = 624, M = 397;

// the 624-word key lives in shared memory; one thread consumes the stream
struct State {
    uint32_t* key;
    int pos, has_gauss;
    double gauss;
};

__device__ inline void seed(State& s, uint32_t x) {
    for (int i = 0; i < N; i++) {
        s.key[i] = x;
        x = 1812433253u * (x ^ (x >> 30)) + (uint32_t)(i + 1);
    }
    s.pos = N; s.has_gauss = 0; s.gauss = 0.0;
}

__device__ __noinline__ void twist(State& s) {
    uint32_t* k = s.key;
    for (int i = 0; i < N; i++) {
        const uint32_t y = (k[i] & 0x80000000u) | (k[(i + 1) % N] & 0x7fffffffu);
        k[i] = k[(i + M) % N] ^ (y >> 1) ^ ((y & 1u) ? 0x9908b0dfu : 0u);
    }
    s.pos = 0;
}

__device__ __forceinline__ uint32_t u32(State& s) {
    if (s.pos == N) twist(s);
    uint32_t y = s.key[s.pos++];
    y ^= y >> 11; y ^= (y << 7) & 0x9d2c5680u; y ^= (y << 15) & 0xefc60000u; y ^= y >> 18;
    return y;
}

__device__ __forceinline__ double dbl(State& s) {
    const int32_t a = (int32_t)(u32(s) >> 5);
    const int32_t b = (int32_t)(u32(s) >> 6);
    return (a * 67108864.0 + b) / 9007199254740992.0;
}

__device__ inline double gauss(State& s) {
    if (s.has_gauss) {
        const double t = s.gauss;
        s.has_gauss = 0; s.gauss = 0.0;
        return t;
    }
    double x1, x2, r2;
    do {
        x1 = 2.0 * dbl(s) - 1.0;
        x2 = 2.0 * dbl(s) - 1.0;
        r2 = x1 * x1 + x2 * x2;
    } while (r2 >= 1.0 || r2 == 0.0);
    const double f = sqrt(-2.0 * log(r2) / r2);
    s.gauss = f * x1; s.has_gauss = 1;
    return f * x2;
}

// pow for the samplers.  CUDA's pow is within 1 ulp for normal results but not in the subnormal range, where Johnk's X / (X + Y)
// then depends on single bits (measured: pow(U, 1 / 7.1e-4) = 0 on the device where glibc gives 2^-1074, so a draw of 0.5 became
// 1.0).  A result below DBL_MIN is recomputed as pow(x, y / 2)^2: the half power is a normal number within 1 ulp, and the one rounding
// of the square into the subnormal grid is the correctly rounded value unless that lies within 2^-51 (relative) of a rounding tie.
// Skipped where x^y <= e^(-y (1 - x)) < e^-750 < 2^-1076 rounds to 0 anyway: the common case pow(U, 1e5) of near-zero steering.
__device__ __noinline__ double pow_np(double x, double y) {
    const double r = pow(x, y);
    if (r < 2.2250738585072014e-308 && y * (1.0 - x) <= 750.0) {
        const double h = pow(x, 0.5 * y);
        return h * h;
    }
    return r;
}

__device__ inline double exponential(State& s) { return -log(1.0 - dbl(s)); }

__device__ __noinline__ double gamma(State& s, double shape) {
    if (shape == 1.0) return exponential(s);
    if (shape == 0.0) return 0.0;
    if (shape < 1.0) {
        for (;;) {
            const double U = dbl(s), V = exponential(s);
            if (U <= 1.0 - shape) {
                const double X = pow_np(U, 1. / shape);
                if (X <= V) return X;
            } else {
                const double Y = -log((1 - U) / shape);
                const double X = pow_np(1.0 - shape + shape * Y, 1. / shape);
                if (X <= (V + Y)) return X;
            }
        }
    }
    const double b = shape - 1. / 3., c = 1. / sqrt(9 * b);
    for (;;) {
        double X, V;
        do {
            X = gauss(s);
            V = 1.0 + c * X;
        } while (V <= 0.0);
        V = V * V * V;
        const double U = dbl(s);
        if (U < 1.0 - 0.0331 * (X * X) * (X * X)) return b * V;
        if (log(U) < 0.5 * X * X + b * (1. - V + log(V))) return b * V;
    }
}

__device__ __noinline__ double beta(State& s, double a, double b) {
    if (a <= 1.0 && b <= 1.0) {                                 // Johnk
        for (;;) {
            const double U = dbl(s), V = dbl(s);
            const double X = pow_np(U, 1.0 / a), Y = pow_np(V, 1.0 / b);
            if ((X + Y) <= 1.0) {
                if (X + Y > 0) return X / (X + Y);
                double lx = log(U) / a, ly = log(V) / b;        // both powers underflowed: log space
                const double lm = lx > ly ? lx : ly;
                lx -= lm; ly -= lm;
                return exp(lx - log(exp(lx) + exp(ly)));
            }
        }
    }
    const double Ga = gamma(s, a), Gb = gamma(s, b);
    return Ga / (Ga + Gb);
}

}  // namespace dnp
