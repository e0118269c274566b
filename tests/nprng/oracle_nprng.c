/* oracle_nprng.c -- C entry points of the legacy-stream restatement (oracle_nprng.h) for the ctypes wrapper in
 * tests/test_validation_rng.py.  TEST INFRASTRUCTURE ONLY.  Build: gcc -O2 -fPIC -shared -ffp-contract=off -fno-fast-math ... -lm.
 *
 * A stream state crosses the ABI as 628 uint32 words, the layout mpcmmd_validate_seeded_host's state_out uses:
 * key[624], pos, has_gauss, then the cached gauss as a float64 bit pattern (low word first). */
#include <string.h>
#include "oracle_nprng.h"

#define NPR_WORDS (NPR_N + 4)

static void unpack(npr_state *s, const uint32_t *w) {
    memcpy(s->key, w, sizeof(s->key));
    s->pos = (int)w[NPR_N]; s->has_gauss = (int)w[NPR_N + 1];
    uint64_t g = (uint64_t)w[NPR_N + 2] | ((uint64_t)w[NPR_N + 3] << 32);
    memcpy(&s->gauss, &g, 8);
}

static void pack(const npr_state *s, uint32_t *w) {
    memcpy(w, s->key, sizeof(s->key));
    w[NPR_N] = (uint32_t)s->pos; w[NPR_N + 1] = (uint32_t)s->has_gauss;
    uint64_t g; memcpy(&g, &s->gauss, 8);
    w[NPR_N + 2] = (uint32_t)g; w[NPR_N + 3] = (uint32_t)(g >> 32);
}

void oracle_npr_seed(uint32_t seed, uint32_t *state) {
    npr_state s; npr_seed(&s, seed); pack(&s, state);
}

/* n draws continuing `state` (updated in place): kind 0 random_sample, 1 standard_normal, 2 standard_exponential,
 * 3 standard_gamma(p1[i]), 4 beta(p1[i], p2[i]) */
void oracle_npr_draw(uint32_t *state, int kind, int n, const double *p1, const double *p2, double *out) {
    npr_state s; unpack(&s, state);
    for (int i = 0; i < n; i++) {
        switch (kind) {
            case 0: out[i] = npr_double(&s); break;
            case 1: out[i] = npr_gauss(&s); break;
            case 2: out[i] = npr_exponential(&s); break;
            case 3: out[i] = npr_gamma(&s, p1[i]); break;
            default: out[i] = npr_beta(&s, p1[i], p2[i]); break;
        }
    }
    pack(&s, state);
}

/* one trajectory's perturbed controls from np.random.seed(seed); state_out: the stream after the last draw */
void oracle_npr_perturbed(uint32_t seed, int noise_kind, int n_roll, int np, const double *acc, const double *steer, double nl, double k_steer,
                          double beta_a, double beta_b, double c_acc, double c_steer, double *acc_out, double *steer_out, uint32_t *state_out) {
    npr_state s; npr_seed(&s, seed);
    npr_perturbed(&s, noise_kind, n_roll, np, acc, steer, nl, k_steer, beta_a, beta_b, c_acc, c_steer, acc_out, steer_out);
    pack(&s, state_out);
}
