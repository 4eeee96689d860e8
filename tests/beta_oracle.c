/*
 * beta_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 * A C restatement of the Beta node of zhusuan-pytorch_b200/csrc/zs_nodes.cu, built by tests/beta_oracle.py
 * (gcc -O2 -ffp-contract=off -shared -fPIC) next to the CPU oracle of oracle/:
 *   - log-density  xlogy(a - 1, x) + xlogy(b - 1, 1 - x) + lgamma(a + b) - (lgamma(a) + lgamma(b)), summed over the
 *     event axis (torch.distributions.Beta.log_prob, via Dirichlet.log_prob), and torch's autograd of it, with
 *     digamma restated from ATen's calc_digamma;
 *   - the sampler on the same Philox words: element i reads its words in order from the Philox4x32-10 groups at
 *     counter i | (j << 48), j = 0, 1, ...; two Marsaglia-Tsang gamma draws (ATen's sample_gamma) in double, normals by
 *     Box-Muller on two words.  glibc and CUDA's double log / cos / pow may differ in the last bit, which can tip an
 *     accept / reject decision: the GPU tests allow a small fraction of disagreeing elements.
 */
#include <float.h>
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

static double next_normal(words_t* u) {
    const double u1 = 1.0 - next_u(u);
    const double u2 = next_u(u);
    return sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
}

static double gamma_draw(double alpha, words_t* u) {
    double scale = 1.0;
    if (alpha < 1.0) {
        scale *= pow(1.0 - next_u(u), 1.0 / alpha);
        alpha += 1.0;
    }
    const double d = alpha - (double)(1.0f / 3.0f);
    const double c = 1.0 / sqrt(9.0 * d);
    while (u->used < MAX_WORDS) {
        const double x = next_normal(u);
        const double y = 1.0 + c * x;
        if (y <= 0.0) continue;
        const double v = y * y * y;
        const double U = 1.0 - next_u(u);
        const double xx = x * x;
        if (U < 1.0 - (double)0.0331f * xx * xx) return scale * d * v;
        if (log(U) < 0.5 * xx + d * (1.0 - v + log(v))) return scale * d * v;
    }
    return scale * d;
}

/* beta_draw_raw: G_a / (G_a + G_b) in double, or NaN for parameters that are not positive and finite */
static double beta_draw_raw(double a, double b, words_t* u) {
    if (!(a > 0.0 && b > 0.0 && a < INFINITY && b < INFINITY)) return NAN;
    const double ga = fmax(gamma_draw(a, u), DBL_MIN);
    const double gb = fmax(gamma_draw(b, u), DBL_MIN);
    return ga / (ga + gb);
}

#define DEFINE(REAL, SFX, LOG, LGAMMA, TRUNC, REAL_MIN, ONE_BELOW)                                                   \
    static REAL ld_##SFX(const REAL* p, int mode, int64_t full_idx, int64_t kb_idx) {                                \
        return mode == FULL ? p[full_idx] : (mode == KBCAST ? p[kb_idx] : p[0]);                                     \
    }                                                                                                                \
    static REAL digamma_##SFX(REAL x) {                                                                              \
        if (x == (REAL)0) return copysign((REAL)INFINITY, -x);                                                       \
        REAL refl = 0;                                                                                               \
        if (x < (REAL)0) {                                                                                           \
            if (x == TRUNC(x)) return (REAL)NAN;                                                                     \
            double q;                                                                                                \
            const double r = modf((double)x, &q);                                                                    \
            refl = (REAL)(3.141592653589793 / tan(3.141592653589793 * r));                                           \
            x = (REAL)1 - x;                                                                                         \
        }                                                                                                            \
        REAL result = 0;                                                                                             \
        while (x < (REAL)10) {                                                                                       \
            result -= (REAL)1 / x;                                                                                   \
            x += (REAL)1;                                                                                            \
        }                                                                                                            \
        if (x == (REAL)10) return (result + (REAL)2.25175258906672110764) - refl;                                    \
        REAL y = 0;                                                                                                  \
        if (x < (REAL)1.0e17) {                                                                                      \
            const REAL z = (REAL)1 / (x * x);                                                                        \
            REAL p = (REAL)8.33333333333333333333E-2;                                                                \
            p = p * z + (REAL)-2.10927960927960927961E-2;                                                            \
            p = p * z + (REAL)7.57575757575757575758E-3;                                                             \
            p = p * z + (REAL)-4.16666666666666666667E-3;                                                            \
            p = p * z + (REAL)3.96825396825396825397E-3;                                                             \
            p = p * z + (REAL)-8.33333333333333333333E-3;                                                            \
            p = p * z + (REAL)8.33333333333333333333E-2;                                                             \
            y = z * p;                                                                                               \
        }                                                                                                            \
        return (((result + LOG(x)) - ((REAL)0.5 / x)) - y) - refl;                                                   \
    }                                                                                                                \
    static REAL xlogy_##SFX(REAL c, REAL v) {                                                                        \
        if (isnan(v)) return v;                                                                                      \
        return c == (REAL)0 ? (REAL)0 : c * LOG(v);                                                                  \
    }                                                                                                                \
    double orc_digamma_##SFX(double x) { return (double)digamma_##SFX((REAL)x); }                                    \
    void orc_beta_sample_##SFX(REAL* out, const REAL* alpha, int am, const REAL* beta, int bm, int64_t K, int64_t N, \
                               uint64_t seed, uint64_t offset) {                                                     \
        for (int64_t i = 0; i < K * N; ++i) {                                                                        \
            words_t u = {(uint64_t)i, offset, seed, {0, 0, 0, 0}, 0};                                                \
            const double r = beta_draw_raw((double)ld_##SFX(alpha, am, i, i % N), (double)ld_##SFX(beta, bm, i, i % N), \
                                           &u);                                                                      \
            if (isnan(r)) {                                                                                          \
                out[i] = (REAL)NAN;                                                                                  \
                continue;                                                                                            \
            }                                                                                                        \
            const REAL v = (REAL)r;                                                                                  \
            out[i] = v < REAL_MIN ? REAL_MIN : (v > ONE_BELOW ? ONE_BELOW : v);                                      \
        }                                                                                                            \
    }                                                                                                                \
    void orc_beta_logprob_fwd_##SFX(REAL* out, const REAL* x, int xm, const REAL* a, int am, const REAL* b, int bm,   \
                                    int64_t K, int64_t M, int64_t E) {                                               \
        for (int64_t k = 0; k < K; ++k)                                                                              \
            for (int64_t m = 0; m < M; ++m) {                                                                        \
                double acc = 0.0;                                                                                    \
                for (int64_t e = 0; e < E; ++e) {                                                                    \
                    const int64_t f = (k * M + m) * E + e, n = m * E + e;                                            \
                    const REAL xv = ld_##SFX(x, xm, f, n), av = ld_##SFX(a, am, f, n), bv = ld_##SFX(b, bm, f, n);   \
                    const REAL s = xlogy_##SFX(av - (REAL)1, xv) + xlogy_##SFX(bv - (REAL)1, (REAL)1 - xv);          \
                    acc += (double)((s + LGAMMA(av + bv)) - (LGAMMA(av) + LGAMMA(bv)));                              \
                }                                                                                                    \
                out[k * M + m] = (REAL)acc;                                                                          \
            }                                                                                                        \
    }                                                                                                                \
    /* each gradient has the layout of its operand (FULL: elementwise, KBCAST: summed over particles); NULL: skip */ \
    void orc_beta_logprob_bwd_##SFX(REAL* dx, REAL* da, REAL* db, const REAL* g, const REAL* x, int xm, const REAL* a, \
                                    int am, const REAL* b, int bm, int64_t K, int64_t M, int64_t E) {                \
        if (dx && xm == KBCAST) for (int64_t n = 0; n < M * E; ++n) dx[n] = (REAL)0;                                 \
        if (da && am == KBCAST) for (int64_t n = 0; n < M * E; ++n) da[n] = (REAL)0;                                 \
        if (db && bm == KBCAST) for (int64_t n = 0; n < M * E; ++n) db[n] = (REAL)0;                                 \
        for (int64_t k = 0; k < K; ++k)                                                                              \
            for (int64_t m = 0; m < M; ++m)                                                                          \
                for (int64_t e = 0; e < E; ++e) {                                                                    \
                    const int64_t f = (k * M + m) * E + e, n = m * E + e;                                            \
                    const REAL gv = g[k * M + m];                                                                    \
                    const REAL xv = ld_##SFX(x, xm, f, n), av = ld_##SFX(a, am, f, n), bv = ld_##SFX(b, bm, f, n);   \
                    const REAL am1 = av - (REAL)1, bm1 = bv - (REAL)1, y = (REAL)1 - xv;                             \
                    const REAL ox = (gv * am1) / xv - (gv * bm1) / y;                                                \
                    const REAL lx = (am1 == (REAL)0 && xv <= (REAL)0) ? (REAL)0 : xlogy_##SFX(gv, xv);               \
                    const REAL ly = (bm1 == (REAL)0 && y <= (REAL)0) ? (REAL)0 : xlogy_##SFX(gv, y);                 \
                    const REAL gs = gv * digamma_##SFX(av + bv);                                                     \
                    const REAL oa = (lx + gs) - gv * digamma_##SFX(av);                                              \
                    const REAL ob = (ly + gs) - gv * digamma_##SFX(bv);                                              \
                    if (dx) { if (xm == KBCAST) dx[n] += ox; else dx[f] = ox; }                                      \
                    if (da) { if (am == KBCAST) da[n] += oa; else da[f] = oa; }                                      \
                    if (db) { if (bm == KBCAST) db[n] += ob; else db[f] = ob; }                                      \
                }                                                                                                    \
    }

DEFINE(float, f32, logf, lgammaf, truncf, FLT_MIN, 0.99999994f)
DEFINE(double, f64, log, lgamma, trunc, DBL_MIN, 0.99999999999999989)
