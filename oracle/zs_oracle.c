/*
 * zs_oracle.c — TEST INFRASTRUCTURE, NOT PRODUCT CODE.  See zs_oracle_impl.h.
 * Build: make -C oracle   (gcc -O2 -fopenmp -ffp-contract=off -shared -fPIC)
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

/* ---- Philox4x32-10 (Salmon, Moraes, Dror, Shaw: "Parallel random numbers: as easy as 1, 2, 3",
 * SC'11), restated from the published algorithm; known-answer vectors from the Random123
 * distribution are checked in tests/test_oracle_golden.py.  Same counter/key convention as the
 * kernels (zhusuan-pytorch_b200/csrc/zs_philox.cuh): counter = (i/4 lo, i/4 hi, offset lo,
 * offset hi), key = (seed lo, seed hi). */
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

/* raw known-answer interface: explicit counter and key */
void orc_philox_kat(uint32_t out[4], const uint32_t ctr[4], const uint32_t key[2]) {
    uint32_t c[4] = {ctr[0], ctr[1], ctr[2], ctr[3]};
    uint32_t k[2] = {key[0], key[1]};
    philox4x32_10(c, k);
    memcpy(out, c, sizeof(c));
}

void orc_philox_raw(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset) {
    for (int64_t q = 0; q < n / 4; ++q) {
        uint32_t c[4] = {(uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
        uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
        philox4x32_10(c, k);
        memcpy(out + 4 * q, c, sizeof(c));
    }
}

static float u01_closed_open(uint32_t r) { return (float)(r >> 8) * 5.9604644775390625e-8f; }
static float u01_open(uint32_t r) { return (float)(r >> 8) * 5.9604644775390625e-8f + 2.98023223876953125e-8f; }

/* ---- per-element word stream of the Poisson and Beta samplers (zhusuan-pytorch_b200/csrc/zs_nodes.cu): element i
 * reads its words in order from the Philox groups at counter i | (j << 48), j = 0, 1, ..., each as a uniform on
 * [0, 1).  A draw gives up after MAX_WORDS words. */
#define MAX_WORDS 256

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
    return (double)u01_closed_open(u->w[u->used++ & 3]);
}

/* Poisson draw with ATen's CPU algorithm (Knuth below rate 10, Hormann's PTRS above) in double.  glibc and CUDA's
 * double log / lgamma may differ in the last bit, which can tip an accept / reject decision: the GPU tests allow a
 * small fraction of disagreeing elements. */
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

/* Beta draw: two Marsaglia-Tsang gamma draws (ATen's sample_gamma) in double, normals by Box-Muller on two words.
 * As for Poisson, libm and CUDA's double log / cos / pow may tip an accept / reject decision. */
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

/* G_a / (G_a + G_b) in double, or NaN for parameters that are not positive and finite */
static double beta_draw_raw(double a, double b, words_t* u) {
    if (!(a > 0.0 && b > 0.0 && a < INFINITY && b < INFINITY)) return NAN;
    const double ga = fmax(gamma_draw(a, u), DBL_MIN);
    const double gb = fmax(gamma_draw(b, u), DBL_MIN);
    return ga / (ga + gb);
}

/* uniforms on the OPEN interval (0,1): the noise source of the Logistic / Laplace samplers */
void orc_philox_uniform_open_f32(float* out, int64_t n, uint64_t seed, uint64_t offset) {
    for (int64_t q = 0; q < (n + 3) / 4; ++q) {
        uint32_t c[4] = {(uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
        uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
        philox4x32_10(c, k);
        for (int j = 0; j < 4; ++j)
            if (4 * q + j < n) out[4 * q + j] = u01_open(c[j]);
    }
}

void orc_philox_uniform_f32(float* out, int64_t n, uint64_t seed, uint64_t offset) {
    for (int64_t q = 0; q < (n + 3) / 4; ++q) {
        uint32_t c[4] = {(uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
        uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
        philox4x32_10(c, k);
        for (int j = 0; j < 4; ++j)
            if (4 * q + j < n) out[4 * q + j] = u01_closed_open(c[j]);
    }
}

/* Box-Muller exactly as zs_philox.cuh: (r0,r1)->(n0,n1), (r2,r3)->(n2,n3) */
void orc_philox_normal_f32(float* out, int64_t n, float mean, float std, uint64_t seed, uint64_t offset) {
    for (int64_t q = 0; q < (n + 3) / 4; ++q) {
        uint32_t c[4] = {(uint32_t)q, (uint32_t)((uint64_t)q >> 32), (uint32_t)offset, (uint32_t)(offset >> 32)};
        uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
        philox4x32_10(c, k);
        float v[4];
        for (int h = 0; h < 2; ++h) {
            float u1 = u01_open(c[2 * h]), u2 = u01_open(c[2 * h + 1]);
            float rad = sqrtf(-2.0f * logf(u1));
            double ang = 2.0 * 3.14159265358979323846 * (double)u2;
            v[2 * h] = rad * (float)cos(ang);
            v[2 * h + 1] = rad * (float)sin(ang);
        }
        for (int j = 0; j < 4; ++j)
            if (4 * q + j < n) out[4 * q + j] = mean + std * v[j];
    }
}

int orc_set_threads(int n) {
#ifdef _OPENMP
    if (n > 0) omp_set_num_threads(n);
    return omp_get_max_threads();
#else
    (void)n;
    return 1;
#endif
}

/* RMIN / RONE_BELOW: the least normal value and the largest value below 1 */
#define REAL float
#define SUFFIX _f32
#define RLOG logf
#define REXP expf
#define RSQRT sqrtf
#define RLGAMMA lgammaf
#define RTRUNC truncf
#define RMIN FLT_MIN
#define RONE_BELOW 0.99999994f
#include "zs_oracle_impl.h"

#define REAL double
#define SUFFIX _f64
#define RLOG log
#define REXP exp
#define RSQRT sqrt
#define RLGAMMA lgamma
#define RTRUNC trunc
#define RMIN DBL_MIN
#define RONE_BELOW 0.99999999999999989
#include "zs_oracle_impl.h"
