/*
 * poisson_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 * A C restatement of the Poisson node of zhusuan-pytorch_b200/csrc/zs_nodes.cu, built by tests/poisson_oracle.py
 * (gcc -O2 -ffp-contract=off -shared -fPIC) next to the CPU oracle of oracle/:
 *   - log-pmf  xlogy(x, rate) - rate - lgamma(x + 1), summed over the event axis, and its rate gradient
 *     g * (x / rate - 1) (torch.distributions.Poisson.log_prob, which the reference's poisson.py:75 calls);
 *   - the sampler on the same Philox words: element i reads its uniforms in order from the Philox4x32-10 groups at
 *     counter i | (j << 48), j = 0, 1, ..., with ATen's CPU algorithm (Knuth below rate 10, Hormann's PTRS above) in
 *     double.  glibc and CUDA's double log / lgamma may differ in the last bit, which can tip an accept / reject
 *     decision: the GPU tests allow a small fraction of disagreeing elements.
 */
#include <math.h>
#include <stdint.h>

enum { FULL = 0, KBCAST = 1, SCALAR = 2 };
#define MAX_WORDS 256

static void philox4x32_10(uint32_t ctr[4], uint32_t key[2]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    uint32_t k0 = key[0], k1 = key[1];
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * ctr[0];
        uint64_t p1 = (uint64_t)M1 * ctr[2];
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ ctr[1] ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ ctr[3] ^ k1;
        uint32_t n3 = (uint32_t)p0;
        ctr[0] = n0; ctr[1] = n1; ctr[2] = n2; ctr[3] = n3;
        k0 += W0; k1 += W1;
    }
}

typedef struct {
    uint64_t i, offset, seed;
    uint32_t w[4];
    int used;
} words_t;

static double next_u(words_t* u) {
    if ((u->used & 3) == 0) {
        const uint64_t ctr = u->i | ((uint64_t)(u->used >> 2) << 48);
        uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)u->offset, (uint32_t)(u->offset >> 32)};
        uint32_t k[2] = {(uint32_t)u->seed, (uint32_t)(u->seed >> 32)};
        philox4x32_10(c, k);
        for (int j = 0; j < 4; ++j) u->w[j] = c[j];
    }
    const uint32_t r = u->w[u->used++ & 3];
    return (double)((float)(r >> 8) * 5.9604644775390625e-8f);
}

static double poisson_draw(double lam, words_t* u) {
    if (lam >= 10.0) {
        const double slam = sqrt(lam), loglam = log(lam);
        const double b = 0.931 + 2.53 * slam;
        const double a = -0.059 + 0.02483 * b;
        const double invalpha = 1.1239 + 1.1328 / (b - 3.4);
        const double vr = 0.9277 - 3.6224 / (b - 2.0);
        while (u->used < MAX_WORDS) {
            const double U = next_u(u) - 0.5;
            const double V = next_u(u);
            const double us = 0.5 - fabs(U);
            const double k = floor((2.0 * a / us + b) * U + lam + 0.43);
            if (us >= 0.07 && V <= vr) return k;
            if (k < 0.0 || (us < 0.013 && V > us)) continue;
            if (log(V) + log(invalpha) - log(a / (us * us) + b) <= -lam + k * loglam - lgamma(k + 1.0)) return k;
        }
        return floor(lam);
    }
    if (lam == 0.0) return 0.0;
    const double enlam = exp(-lam);
    double x = 0.0, prod = 1.0;
    while (u->used < MAX_WORDS) {
        prod *= next_u(u);
        if (!(prod > enlam)) return x;
        x += 1.0;
    }
    return x;
}

#define DEFINE(REAL, SFX, LOG, LGAMMA)                                                                              \
    static REAL ld_##SFX(const REAL* p, int mode, int64_t full_idx, int64_t kb_idx) {                                \
        return mode == FULL ? p[full_idx] : (mode == KBCAST ? p[kb_idx] : p[0]);                                     \
    }                                                                                                                \
    void orc_poisson_sample_##SFX(REAL* out, const REAL* rate, int rm, int64_t K, int64_t N, uint64_t seed,          \
                                  uint64_t offset) {                                                                 \
        for (int64_t i = 0; i < K * N; ++i) {                                                                        \
            words_t u = {(uint64_t)i, offset, seed, {0, 0, 0, 0}, 0};                                                \
            out[i] = (REAL)poisson_draw((double)ld_##SFX(rate, rm, i, i % N), &u);                                   \
        }                                                                                                            \
    }                                                                                                                \
    void orc_poisson_logpmf_fwd_##SFX(REAL* out, const REAL* x, int xm, const REAL* rate, int rm, int64_t K,         \
                                      int64_t M, int64_t E) {                                                        \
        for (int64_t k = 0; k < K; ++k)                                                                              \
            for (int64_t m = 0; m < M; ++m) {                                                                        \
                double acc = 0.0;                                                                                    \
                for (int64_t e = 0; e < E; ++e) {                                                                    \
                    const int64_t f = (k * M + m) * E + e, n = m * E + e;                                            \
                    const REAL xv = ld_##SFX(x, xm, f, n), r = ld_##SFX(rate, rm, f, n);                             \
                    const REAL xl = (xv == (REAL)0 && !isnan(r)) ? (REAL)0 : xv * LOG(r);                            \
                    acc += (double)((xl - r) - LGAMMA(xv + (REAL)1));                                                \
                }                                                                                                    \
                out[k * M + m] = (REAL)acc;                                                                          \
            }                                                                                                        \
    }                                                                                                                \
    /* drate has the layout of `rate` (FULL: elementwise, KBCAST: summed over particles) */                         \
    void orc_poisson_logpmf_bwd_##SFX(REAL* drate, const REAL* g, const REAL* x, int xm, const REAL* rate, int rm,   \
                                      int64_t K, int64_t M, int64_t E) {                                             \
        if (rm == KBCAST)                                                                                            \
            for (int64_t n = 0; n < M * E; ++n) drate[n] = (REAL)0;                                                  \
        for (int64_t k = 0; k < K; ++k)                                                                              \
            for (int64_t m = 0; m < M; ++m)                                                                          \
                for (int64_t e = 0; e < E; ++e) {                                                                    \
                    const int64_t f = (k * M + m) * E + e, n = m * E + e;                                           \
                    const REAL xv = ld_##SFX(x, xm, f, n), r = ld_##SFX(rate, rm, f, n);                             \
                    const REAL d = g[k * M + m] * (xv / r - (REAL)1);                                                \
                    if (rm == KBCAST) drate[n] += d;                                                                 \
                    else drate[f] = d;                                                                               \
                }                                                                                                    \
    }

DEFINE(float, f32, logf, lgammaf)
DEFINE(double, f64, log, lgamma)
