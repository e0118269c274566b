// drng.cuh -- device restatement of the JAX 0.3.23 PRNG protocol used by the reference
// (jax is a third-party dependency of the reference, pinned jax==0.3.23 in requirements.txt:1):
// Threefry-2x32 counter RNG, random.split / bits / uniform / normal and the Marsaglia-Tsang
// log-space gamma sampler behind random.beta.  Reference call sites:
//   S/optimizer/cem.py:225,254,302   S/optimizer/cem_helper.py:125-126,405-443,470-508
//   S/compute_beta.py:25,44,54,108,131
// All transcendental arithmetic goes through dmath.cuh (deterministic contract).
#pragma once
#include "dmath.cuh"

namespace dr {

struct Key { uint32_t k0, k1; };

__device__ __forceinline__ uint32_t rotl(uint32_t x, int d) { return (x << d) | (x >> (32 - d)); }

__device__ __noinline__ void threefry2x32(Key key, uint32_t x0, uint32_t x1, uint32_t& o0, uint32_t& o1) {
    const uint32_t ks0 = key.k0, ks1 = key.k1, ks2 = key.k0 ^ key.k1 ^ 0x1BD11BDAu;
    x0 += ks0; x1 += ks1;
#define TF_R(r) { x0 += x1; x1 = rotl(x1, r); x1 ^= x0; }
    TF_R(13) TF_R(15) TF_R(26) TF_R(6)   x0 += ks1; x1 += ks2 + 1u;
    TF_R(17) TF_R(29) TF_R(16) TF_R(24)  x0 += ks2; x1 += ks0 + 2u;
    TF_R(13) TF_R(15) TF_R(26) TF_R(6)   x0 += ks0; x1 += ks1 + 3u;
    TF_R(17) TF_R(29) TF_R(16) TF_R(24)  x0 += ks1; x1 += ks2 + 4u;
    TF_R(13) TF_R(15) TF_R(26) TF_R(6)   x0 += ks2; x1 += ks0 + 5u;
#undef TF_R
    o0 = x0; o1 = x1;
}

// element i of random_bits(key, 32, (n,)): counters iota(n) padded to even, first half / second
// half form the two Threefry words, outputs concatenated.
__device__ __forceinline__ uint32_t bits_elem(Key key, uint32_t n, uint32_t i) {
    const uint32_t half = (n + (n & 1u)) >> 1;
    uint32_t c0, c1, a, b;
    if (i < half) { c0 = i; c1 = i + half; if (c1 >= n) c1 = 0u; }
    else { c0 = i - half; c1 = i; }
    threefry2x32(key, c0, c1, a, b);
    return (i < half) ? a : b;
}
// row r of random.split(key, m) = bits(key, 2m).reshape(m, 2)
__device__ __forceinline__ Key split_row(Key key, uint32_t m, uint32_t r) {
    Key o;
    o.k0 = bits_elem(key, 2u * m, 2u * r);
    o.k1 = bits_elem(key, 2u * m, 2u * r + 1u);
    return o;
}
// key, _ = split(key): bits(key,4) = [a0,a1,b0,b1] with (a0,b0)=tf(0,2), (a1,b1)=tf(1,3); row 0 = (a0,a1)
__device__ __forceinline__ Key split0(Key key) {
    uint32_t a0, b0, a1, b1;
    threefry2x32(key, 0u, 2u, a0, b0);
    threefry2x32(key, 1u, 3u, a1, b1);
    Key o; o.k0 = a0; o.k1 = a1;
    return o;
}
__device__ __forceinline__ void split2(Key key, Key& r0, Key& r1) {
    uint32_t a0, b0, a1, b1;
    threefry2x32(key, 0u, 2u, a0, b0);
    threefry2x32(key, 1u, 3u, a1, b1);
    r0.k0 = a0; r0.k1 = a1; r1.k0 = b0; r1.k1 = b1;
}
// split(key, 3): bits(key, 6): half = 3: tf(0,3),tf(1,4),tf(2,5) -> [a0,a1,a2,b0,b1,b2] -> rows (a0,a1),(a2,b0),(b1,b2)
__device__ __forceinline__ void split3(Key key, Key& r0, Key& r1, Key& r2) {
    uint32_t a0, b0, a1, b1, a2, b2;
    threefry2x32(key, 0u, 3u, a0, b0);
    threefry2x32(key, 1u, 4u, a1, b1);
    threefry2x32(key, 2u, 5u, a2, b2);
    r0.k0 = a0; r0.k1 = a1; r1.k0 = a2; r1.k1 = b0; r2.k0 = b1; r2.k1 = b2;
}
__device__ __forceinline__ uint32_t bits1(Key key) { uint32_t a, b; threefry2x32(key, 0u, 0u, a, b); return a; }

__device__ __forceinline__ float bits_to_unit(uint32_t b) { return dm::u2f((b >> 9) | 0x3F800000u) - 1.0f; }

// XLA ErfInv (float32): Giles' polynomial in w = -log1p(-x*x)
__device__ __forceinline__ float erfinv32(float x) {
    if (fabsf(x) == 1.0f) return x * DM_INF;
    float xx = x * x;
    float w = -dm::log1p_(-xx);
    float p;
    if (w < 5.0f) {
        w = w - 2.5f;
        p = 2.81022636e-08f;
        p = 3.43273939e-07f + p * w;
        p = -3.5233877e-06f + p * w;
        p = -4.39150654e-06f + p * w;
        p = 0.00021858087f + p * w;
        p = -0.00125372503f + p * w;
        p = -0.00417768164f + p * w;
        p = 0.246640727f + p * w;
        p = 1.50140941f + p * w;
    } else {
        w = sqrtf(w) - 3.0f;
        p = -0.000200214257f;
        p = 0.000100950558f + p * w;
        p = 0.00134934322f + p * w;
        p = -0.00367342844f + p * w;
        p = 0.00573950773f + p * w;
        p = -0.0076224613f + p * w;
        p = 0.00943887047f + p * w;
        p = 1.00167406f + p * w;
        p = 2.83297682f + p * w;
    }
    return p * x;
}
// uniform(minval=lo, maxval=1) with lo = nextafter(-1, 0), then sqrt(2)*erfinv: one normal from 32 bits
__device__ __forceinline__ float normal_from_bits(uint32_t b) {
    const float lo = -0.99999994f;               // nextafterf(-1, 0)
    float t = bits_to_unit(b) * (1.0f - lo);
    float v = t + lo;
    v = v > lo ? v : lo;
    return 1.41421354f * erfinv32(v);            // (float)sqrt(2)
}
__device__ __forceinline__ float uniform01_from_bits(uint32_t b) {
    float v = bits_to_unit(b) * 1.0f + 0.0f;
    return v > 0.0f ? v : 0.0f;
}
__device__ __forceinline__ float normal_elem(Key key, uint32_t n, uint32_t i) { return normal_from_bits(bits_elem(key, n, i)); }

// jax/_src/random.py::_gamma_one(key, alpha, log_space=True): log of a Gamma(alpha,1) sample.
__device__ __noinline__ float loggamma_one(Key key, float alpha) {
    const float one_over_three = 0.333333343f, squeeze_const = 0.0331f;
    const bool boost_mask = alpha >= 1.0f;
    const float alpha_orig = alpha;
    alpha = boost_mask ? alpha : alpha + 1.0f;
    const float d = alpha - one_over_three;
    const float c = one_over_three / sqrtf(d);
    Key subkey;
    { Key k0; split2(key, k0, subkey); key = k0; }
    float X = 0.0f, V = 1.0f, U = 2.0f;
    for (;;) {
        float xx = squeeze_const * (X * X);
        bool c1 = U >= 1.0f - xx;
        float t1 = X * 0.5f, t2 = d * ((1.0f - V) + dm::log_(V));
        bool c2 = dm::log_(U) >= t1 + t2;
        if (!(c1 && c2)) break;
        Key xk, uk;
        { Key k0; split3(key, k0, xk, uk); key = k0; }
        float x = 0.0f, v = -1.0f;
        while (v <= 0.0f) {
            Key s0, s1; split2(xk, s0, s1);
            xk = s0;
            x = normal_from_bits(bits1(s1));
            float xc = x * c;
            v = 1.0f + xc;
        }
        X = x * x;
        float vv = v * v;
        V = vv * v;
        U = uniform01_from_bits(bits1(uk));
    }
    float u = uniform01_from_bits(bits1(subkey));
    float log_samples = -(-dm::log1p_(-u));
    float log_boost;
    if (boost_mask || log_samples == 0.0f) log_boost = 0.0f;
    else log_boost = log_samples * (1.0f / alpha_orig);
    return (dm::log_(d) + dm::log_(V)) + log_boost;
}
// element e (of n) of random.beta(key, a, b, shape) with already-broadcast parameters
__device__ __noinline__ float beta_elem(Key key, uint32_t n, uint32_t e, float a, float b) {
    Key ka, kb; split2(key, ka, kb);
    float lga = loggamma_one(split_row(ka, n, e), a);
    float lgb = loggamma_one(split_row(kb, n, e), b);
    float m = lga > lgb ? lga : lgb;
    if (lga != lga || lgb != lgb) m = DM_NAN;
    float ga = dm::exp_(lga - m), gb = dm::exp_(lgb - m);
    return ga / (ga + gb);
}
// beta_elem with (ka, kb) = split(key) made by the caller: a stream drawn element by element splits its key once, not per element
__device__ __noinline__ float beta_elem_split(Key ka, Key kb, uint32_t n, uint32_t e, float a, float b) {
    float lga = loggamma_one(split_row(ka, n, e), a);
    float lgb = loggamma_one(split_row(kb, n, e), b);
    float m = lga > lgb ? lga : lgb;
    if (lga != lga || lgb != lgb) m = DM_NAN;
    float ga = dm::exp_(lga - m), gb = dm::exp_(lgb - m);
    return ga / (ga + gb);
}

// ---------------------------------------------------------------------------------------------
// Replay form of the Beta sampler.  Every random number _gamma_one consumes is a pure function of (element key, round r,
// inner try j) -- the Gamma parameter only decides which of them are accepted -- and the reference gives all num_batch
// samples of an episode the SAME key (cem_helper.py:109-110, in_axes=(0,0,None,None)).  So the candidates are drawn once per
// (episode, iteration, element) into a table (gamma_table_fill, ~30 Threefry calls) and each of the 100 samples replays the
// acceptance test on them (loggamma_replay: 2 logs, no Threefry).  The table holds rounds 0..2 (and a second inner try for
// round 0); a sample that needs more (probability ~5e-4) falls back to loggamma_one.  Bit-identical to beta_elem.
#define GT_FIELDS 11   // x00, x01, U0, logU0, x10, U1, logU1, x20, U2, logU2, log1p(-u_boost)

// stream: 0/1 = (ka, kb) of the acceleration key, 2/3 = (ka, kb) of the steering key
__device__ __forceinline__ Key gamma_stream_key(Key k_acc, Key k_steer, int stream) {
    Key ka, kb; split2(stream < 2 ? k_acc : k_steer, ka, kb);
    return (stream & 1) ? kb : ka;
}
__device__ __forceinline__ void gamma_table_fill(Key stream_key, uint32_t n, uint32_t e, float* t /* field f at t[f*n] */) {
    Key key = split_row(stream_key, n, e);
    Key subkey;
    { Key k0; split2(key, k0, subkey); key = k0; }
#pragma unroll 1
    for (int r = 0; r < 3; r++) {
        Key xk, uk;
        { Key k0; split3(key, k0, xk, uk); key = k0; }
        Key s0, s1; split2(xk, s0, s1);
        const int base = r == 0 ? 0 : (r == 1 ? 4 : 7);
        t[(size_t)base * n] = normal_from_bits(bits1(s1));
        int fu = base + 1;
        if (r == 0) { Key s0b, s1b; split2(s0, s0b, s1b); t[(size_t)1 * n] = normal_from_bits(bits1(s1b)); fu = 2; }
        const float U = uniform01_from_bits(bits1(uk));
        t[(size_t)fu * n] = U; t[(size_t)(fu + 1) * n] = dm::log_(U);
    }
    const float u = uniform01_from_bits(bits1(subkey));
    t[(size_t)10 * n] = dm::log1p_(-u);
}
// PF (latency regime): all eleven candidate fields are requested up front, so a replay costs ONE global-memory round trip instead of up to four dependent ones
// (the acceptance test decides which fields it reads); the throughput kernels keep the lazy loads (most samples accept in round 0 and read five fields).
template <bool PF = false>
__device__ __forceinline__ float loggamma_replay(const float* __restrict__ t, size_t n, float alpha, bool& ok) {
    float pf[GT_FIELDS];
    if constexpr (PF) {
#pragma unroll
        for (int i = 0; i < GT_FIELDS; i++) pf[i] = t[(size_t)i * n];
    }
    auto T = [&](int i) -> float { if constexpr (PF) return pf[i]; else return t[(size_t)i * n]; };
    const float one_over_three = 0.333333343f, squeeze_const = 0.0331f;
    const bool boost_mask = alpha >= 1.0f;
    const float alpha_orig = alpha;
    alpha = boost_mask ? alpha : alpha + 1.0f;
    const float d = alpha - one_over_three;
    const float c = one_over_three / sqrtf(d);
    float x = T(0);
    float v = 1.0f + x * c;
    if (v <= 0.0f) { x = T(1); v = 1.0f + x * c; if (v <= 0.0f) ok = false; }
    float X = x * x, V = (v * v) * v, lv = dm::log_(V);
    bool cont;
    { const float U = T(2), LU = T(3); const float xx = squeeze_const * (X * X); cont = (U >= 1.0f - xx) && (LU >= X * 0.5f + d * ((1.0f - V) + lv)); }
    if (cont) {
        x = T(4); v = 1.0f + x * c; if (v <= 0.0f) ok = false;
        X = x * x; V = (v * v) * v; lv = dm::log_(V);
        { const float U = T(5), LU = T(6); const float xx = squeeze_const * (X * X); cont = (U >= 1.0f - xx) && (LU >= X * 0.5f + d * ((1.0f - V) + lv)); }
        if (cont) {
            x = T(7); v = 1.0f + x * c; if (v <= 0.0f) ok = false;
            X = x * x; V = (v * v) * v; lv = dm::log_(V);
            { const float U = T(8), LU = T(9); const float xx = squeeze_const * (X * X); cont = (U >= 1.0f - xx) && (LU >= X * 0.5f + d * ((1.0f - V) + lv)); }
            if (cont) ok = false;
        }
    }
    const float lb = T(10);
    float log_boost;
    if (boost_mask || lb == 0.0f) log_boost = 0.0f;
    else log_boost = lb * (1.0f / alpha_orig);
    return (dm::log_(d) + lv) + log_boost;
}
// element e of random.beta(key, a, b): tab -> [2 streams (a, b)][GT_FIELDS][n]; (ka, kb) = split(key) for the fallback
template <bool PF = false>
__device__ __forceinline__ float beta_replay(const float* __restrict__ tab, Key key, uint32_t n, uint32_t e, float a, float b) {
    bool oka = true, okb = true;
    float lga = loggamma_replay<PF>(tab + e, n, a, oka);
    float lgb = loggamma_replay<PF>(tab + (size_t)GT_FIELDS * n + e, n, b, okb);
    if (!(oka && okb)) {                       // rare: more candidates needed than the table holds
        Key ka, kb; split2(key, ka, kb);
        if (!oka) lga = loggamma_one(split_row(ka, n, e), a);
        if (!okb) lgb = loggamma_one(split_row(kb, n, e), b);
    }
    float m = lga > lgb ? lga : lgb;
    if (lga != lga || lgb != lgb) m = DM_NAN;
    float ga = dm::exp_(lga - m), gb = dm::exp_(lgb - m);
    return ga / (ga + gb);
}

}  // namespace dr
