// Stochastic-node kernels: sample and log-prob (forward / backward) for Normal, Bernoulli, Poisson and Beta
// over the [K, M, E] particle-row view described in include/zs_b200.h.
//
// Replaces (reference file:line):
//   Normal._sample        zhusuan/distributions/normal.py:89-107
//   Normal._log_prob      zhusuan/distributions/normal.py:109-126
//   Bernoulli._sample     zhusuan/distributions/bernoulli.py:72-82
//   Bernoulli._log_prob   zhusuan/distributions/bernoulli.py:84-95
//   Distribution.log_prob zhusuan/distributions/base.py:161-178      (group_ndims sum)
//   StochasticTensor.log_prob  zhusuan/framework/stochastic_tensor.py:160-181 (trailing sums)
// The `.repeat([K,1,...])` of the parameters is replaced by the ZS_KBCAST operand mode, the
// CPU-side RNG + H2D copy by in-kernel Philox, and the ~8 (fwd) / ~12 (bwd) elementwise aten
// kernels plus the event-axis reduction by one pass each.
#include "zs_common.cuh"

#include <cooperative_groups.h>
#include <float.h>
#include <type_traits>
#include "zs_philox.cuh"

namespace zs {

// ---------------------------------------------------------------------------
// operand addressing
// ---------------------------------------------------------------------------
template <typename T>
struct Operand {
    const T* p;
    int mode;
    // base pointer of row r = k*M + m (E elements); SCALAR rows are handled by the caller
    __device__ __forceinline__ const T* row(int64_t r, int64_t m, int64_t E) const {
        return mode == ZS_FULL ? p + r * E : p + m * E;
    }
};

// ---------------------------------------------------------------------------
// per-element math
// ---------------------------------------------------------------------------
template <typename T>
struct NormalOp {
    // normal.py:122: a 0-d float64 tensor, rounded to the operand dtype when combined
    static __device__ __forceinline__ T c() { return (T)(-0.9189385332046727); }
    static __device__ __forceinline__ T term(T x, T mean, T std) {
        T logstd = Real<T>::log(std);
        T prec = Real<T>::exp(T(-2) * logstd);
        T d = x - mean;
        return (c() - logstd) - (T(0.5) * prec) * (d * d);
    }
    static __device__ __forceinline__ T finish(T acc) { return acc; }
    // autograd of the expression above, same association order
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(T g, T x, T mean, T std, T& dx, T& dmean, T& dstd) {
        T logstd = Real<T>::log(std);
        T prec = Real<T>::exp(T(-2) * logstd);
        T d = x - mean;
        T dd = -(g * (T(0.5) * prec)) * (T(2) * d);
        dx = dd;
        dmean = -dd;
        T dprec = -(g * (d * d)) * T(0.5);
        T dlogstd = -g + (dprec * prec) * T(-2);
        dstd = dlogstd / std;
    }
};

// Laplace(loc, scale): torch.distributions.Laplace.log_prob as the reference calls it
// (zhusuan/distributions/laplace.py:92): -log(2 scale) - |x - loc| / scale
template <typename T>
struct LaplaceOp {
    static __device__ __forceinline__ T term(T x, T loc, T scale) {
        T d = x - loc;
        return -Real<T>::log(T(2) * scale) - (d < T(0) ? -d : d) / scale;
    }
    static __device__ __forceinline__ T finish(T acc) { return acc; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(T g, T x, T loc, T scale, T& dx, T& dloc, T& dscale) {
        T d = x - loc;
        T sg = d > T(0) ? T(1) : (d < T(0) ? T(-1) : T(0));  // torch: d|u|/du = sign(u), 0 at u = 0
        T ad = d < T(0) ? -d : d;
        dx = -(g * sg) / scale;
        dloc = -dx;
        dscale = -g / scale + (g * ad) / (scale * scale);
    }
};

// Uniform(low, high): torch.distributions.Uniform.log_prob as the reference calls it (zhusuan/distributions/uniform.py:81):
//   log(1[low <= x] * 1[x < high]) - log(high - low), i.e. -log(high - low) inside the support and -inf outside;
// autograd sees only the second term: d/dlow = +g/(high - low), d/dhigh = -g/(high - low), d/dx = 0.
template <typename T>
struct UniformOp {
    static __device__ __forceinline__ T term(T x, T low, T high) {
        const T inside = (low <= x && x < high) ? T(0) : -INFINITY;
        return inside - Real<T>::log(high - low);
    }
    static __device__ __forceinline__ T finish(T acc) { return acc; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(T g, T x, T low, T high, T& dx, T& dlow, T& dhigh) {
        const T r = g / (high - low);
        dx = T(0);
        dlow = r;
        dhigh = -r;
    }
};

// Logistic(loc, scale): zhusuan/distributions/logistic.py:81-82
//   z = (x - loc) / scale ;  log p = -z - 2 softplus(-z) - log(scale)      (softplus: torch's, threshold 20)
template <typename T>
struct LogisticOp {
    static __device__ __forceinline__ T softplus(T v) { return v > T(20) ? v : log1p(Real<T>::exp(v)); }
    static __device__ __forceinline__ T term(T x, T loc, T scale) {
        T z = (x - loc) / scale;
        return (-z - T(2) * softplus(-z)) - Real<T>::log(scale);
    }
    static __device__ __forceinline__ T finish(T acc) { return acc; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(T g, T x, T loc, T scale, T& dx, T& dloc, T& dscale) {
        T z = (x - loc) / scale;
        // d/dz(-z - 2 softplus(-z)) = -1 + 2 sigmoid(-z)   (softplus' = sigmoid below the threshold, 1 above)
        T sgm = -z > T(20) ? T(1) : T(1) / (T(1) + Real<T>::exp(z));
        T dz = g * (T(-1) + T(2) * sgm);
        dx = dz / scale;
        dloc = -dx;
        dscale = -(dz * z) / scale - g / scale;
    }
};

template <typename T>
struct BernoulliOp;

template <>
struct BernoulliOp<float> {
    // accumulate in log2 units on the SFU, scale by ln2 once per row
    static __device__ __forceinline__ float term(float x, float p, float) {
        float a = p + 1e-8f;
        float b = (1.0f - p) + 1e-8f;
        return x * fast_log2(a) + (1.0f - x) * fast_log2(b);
    }
    static __device__ __forceinline__ float finish(float acc) { return acc * 0.6931471805599453f; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(float g, float x, float p, float, float& dx, float& dp, float& unused) {
        float a = p + 1e-8f;
        float b = (1.0f - p) + 1e-8f;
        dp = __fdividef(g * x, a) - __fdividef(g * (1.0f - x), b);
        if (NEED_X) dx = g * ((fast_log2(a) - fast_log2(b)) * 0.6931471805599453f);
        unused = 0.f;
    }
};
template <>
struct BernoulliOp<double> {
    static __device__ __forceinline__ double term(double x, double p, double) {
        return x * ::log(p + 1e-8) + (1.0 - x) * ::log((1.0 - p) + 1e-8);
    }
    static __device__ __forceinline__ double finish(double acc) { return acc; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(double g, double x, double p, double, double& dx, double& dp,
                                                double& unused) {
        double a = p + 1e-8, b = (1.0 - p) + 1e-8;
        dp = (g * x) / a - (g * (1.0 - x)) / b;
        if (NEED_X) dx = g * (::log(a) - ::log(b));
        unused = 0.0;
    }
};

// Bernoulli parameterised by logits (bernoulli.py:47-50 builds probs = sigmoid(logits) and then evaluates the same
// log-pmf, :84-95): the sigmoid is computed in registers, so the decoder's final Sigmoid and its backward never make
// a round trip through HBM (SURVEY 8(f)-1).  Same "+1e-8" arguments as the probs form; d/dlogits = d/dp * p (1 - p).
template <typename T>
struct BernoulliLogitsOp;

template <>
struct BernoulliLogitsOp<float> {
    static __device__ __forceinline__ float sigmoid(float l) { return fast_sigmoid(l); }
    static __device__ __forceinline__ float term(float x, float l, float) {
        return BernoulliOp<float>::term(x, sigmoid(l), 0.f);
    }
    static __device__ __forceinline__ float finish(float acc) { return acc * 0.6931471805599453f; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(float g, float x, float l, float, float& dx, float& dl, float& unused) {
        const float p = sigmoid(l);
        float dp;
        BernoulliOp<float>::grad<NEED_X>(g, x, p, 0.f, dx, dp, unused);
        dl = dp * ((1.0f - p) * p);
    }
};
template <>
struct BernoulliLogitsOp<double> {
    static __device__ __forceinline__ double sigmoid(double l) { return 1.0 / (1.0 + ::exp(-l)); }
    static __device__ __forceinline__ double term(double x, double l, double) {
        return BernoulliOp<double>::term(x, sigmoid(l), 0.0);
    }
    static __device__ __forceinline__ double finish(double acc) { return acc; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(double g, double x, double l, double, double& dx, double& dl,
                                                double& unused) {
        const double p = sigmoid(l);
        double dp;
        BernoulliOp<double>::grad<NEED_X>(g, x, p, 0.0, dx, dp, unused);
        dl = dp * ((1.0 - p) * p);
    }
};

__device__ __forceinline__ float lgamma_t(float v) { return lgammaf(v); }
__device__ __forceinline__ double lgamma_t(double v) { return ::lgamma(v); }

// Poisson(rate): torch.distributions.Poisson.log_prob, which the reference's Poisson._log_prob calls
// (zhusuan/distributions/poisson.py:75):  xlogy(x, rate) - rate - lgamma(x + 1).
// xlogy is 0 at x == 0 unless rate is NaN, so rate == 0 gives 0 at x == 0 and -inf at x > 0.
// d/drate = g (x / rate - 1), torch's xlogy backward; the count carries no gradient (the host refuses one).
template <typename T>
struct PoissonOp {
    static __device__ __forceinline__ T term(T x, T rate, T) {
        const T xl = (x == T(0) && !isnan(rate)) ? T(0) : x * Real<T>::log(rate);
        return (xl - rate) - lgamma_t(x + T(1));
    }
    static __device__ __forceinline__ T finish(T acc) { return acc; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(T g, T x, T rate, T, T& dx, T& drate, T& unused) {
        drate = g * (x / rate - T(1));
        dx = T(0);
        unused = T(0);
    }
};

// digamma, restating ATen's calc_digamma (ATen/native/Math.h, from Cephes): the reflection for x < 0, the recurrence
// up to 10, PSI_10 at exactly 10, the asymptotic series above.  The float form stays in float except for the
// reflection term, as ATen's CPU float version does.
template <typename T>
__device__ __forceinline__ T digamma_t(T x) {
    if (x == T(0)) return copysign((T)INFINITY, -x);
    T refl = T(0);
    if (x < T(0)) {
        if (x == trunc(x)) return (T)NAN;
        double q;
        const double r = modf((double)x, &q);
        refl = (T)(3.141592653589793 / ::tan(3.141592653589793 * r));
        x = T(1) - x;
    }
    T result = T(0);
    while (x < T(10)) {
        result -= T(1) / x;
        x += T(1);
    }
    if (x == T(10)) return (result + (T)2.25175258906672110764) - refl;
    T y = T(0);
    if (x < (T)1.0e17) {
        const T z = T(1) / (x * x);
        T p = (T)8.33333333333333333333E-2;
        p = p * z + (T)-2.10927960927960927961E-2;
        p = p * z + (T)7.57575757575757575758E-3;
        p = p * z + (T)-4.16666666666666666667E-3;
        p = p * z + (T)3.96825396825396825397E-3;
        p = p * z + (T)-8.33333333333333333333E-3;
        p = p * z + (T)8.33333333333333333333E-2;
        y = z * p;
    }
    return (((result + Real<T>::log(x)) - (T(0.5) / x)) - y) - refl;
}

// Beta(alpha, beta): torch.distributions.Beta.log_prob, which goes through Dirichlet.log_prob on stack([x, 1 - x]):
//   xlogy(alpha - 1, x) + xlogy(beta - 1, 1 - x) + lgamma(alpha + beta) - (lgamma(alpha) + lgamma(beta))
// with 1 - x rounded in the operand dtype first, as torch does.  Gradients are torch's autograd of that expression:
//   dx = g (alpha - 1) / x - g (beta - 1) / (1 - x),  dalpha = xlogy(g, x) + g psi(alpha + beta) - g psi(alpha)
// with xlogy's rule that drops the log where alpha - 1 == 0 and x <= 0 (and likewise for beta and 1 - x).
// The parameter-only terms (the two lgamma sums; the three psi values) come in as arguments, so that a caller holding
// them for many elements (ScalarB, k_kreduce_bwd_hoisted) computes bit-identically to term / grad.
template <typename T>
struct BetaOp {
    static __device__ __forceinline__ T xlogy(T c, T v) {
        if (isnan(v)) return v;
        return c == T(0) ? T(0) : c * Real<T>::log(v);
    }
    static __device__ __forceinline__ T lgab(T a, T b) { return lgamma_t(a + b); }
    static __device__ __forceinline__ T lga_lgb(T a, T b) { return lgamma_t(a) + lgamma_t(b); }
    static __device__ __forceinline__ T term_h(T x, T a, T b, T lab, T la_lb) {
        const T s = xlogy(a - T(1), x) + xlogy(b - T(1), T(1) - x);
        return (s + lab) - la_lb;
    }
    static __device__ __forceinline__ T term(T x, T a, T b) { return term_h(x, a, b, lgab(a, b), lga_lgb(a, b)); }
    static __device__ __forceinline__ T finish(T acc) { return acc; }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad_h(T g, T x, T a, T b, T psab, T psa, T psb, T& dx, T& da, T& db) {
        const T am1 = a - T(1), bm1 = b - T(1), y = T(1) - x;
        dx = NEED_X ? (g * am1) / x - (g * bm1) / y : T(0);
        const T lx = (am1 == T(0) && x <= T(0)) ? T(0) : xlogy(g, x);
        const T ly = (bm1 == T(0) && y <= T(0)) ? T(0) : xlogy(g, y);
        const T gs = g * psab;
        da = (lx + gs) - g * psa;
        db = (ly + gs) - g * psb;
    }
    template <bool NEED_X>
    static __device__ __forceinline__ void grad(T g, T x, T a, T b, T& dx, T& da, T& db) {
        grad_h<NEED_X>(g, x, a, b, digamma_t(a + b), digamma_t(a), digamma_t(b), dx, da, db);
    }
};

// ---------------------------------------------------------------------------
// A SCALAR (or absent) second parameter is the same for every element of the launch: whatever the op derives from it
// alone is computed once per thread, not once per element.  For the Normal op that is log(std), exp(-2 log std) and
// 1/std -- the BNN likelihood of bnn_vi.py:55-60 (mean [K, batch], ONE logstd) otherwise spends three transcendentals
// per element on a constant and is issue-bound at 0.3-0.4 of the HBM roofline (profiles/r1_bnn_kernels.json).
// Same expressions in the same order as Op::term / Op::grad, so results are bit-identical.
// `a_` / `a_scalar`: the first parameter, for ops whose parameter-only terms need both (Beta, when both are SCALAR).
// ---------------------------------------------------------------------------
template <typename T, typename Op>
struct ScalarB {
    T b;
    __device__ __forceinline__ ScalarB(T b_, T /*a_*/, bool /*a_scalar*/) : b(b_) {}
    __device__ __forceinline__ T term(T x, T a) const { return Op::term(x, a, b); }
    template <bool NEED_X>
    __device__ __forceinline__ void grad(T g, T x, T a, T& dx, T& da, T& db) const {
        Op::template grad<NEED_X>(g, x, a, b, dx, da, db);
    }
};
template <typename T>
struct ScalarB<T, NormalOp<T>> {
    T std, logstd, prec;
    __device__ __forceinline__ ScalarB(T b_, T /*a_*/, bool /*a_scalar*/) : std(b_) {
        logstd = Real<T>::log(b_);
        prec = Real<T>::exp(T(-2) * logstd);
    }
    __device__ __forceinline__ T term(T x, T mean) const {
        T d = x - mean;
        return (NormalOp<T>::c() - logstd) - (T(0.5) * prec) * (d * d);
    }
    template <bool NEED_X>
    __device__ __forceinline__ void grad(T g, T x, T mean, T& dx, T& dmean, T& dstd) const {
        T d = x - mean;
        T dd = -(g * (T(0.5) * prec)) * (T(2) * d);
        dx = dd;
        dmean = -dd;
        T dprec = -(g * (d * d)) * T(0.5);
        T dlogstd = -g + (dprec * prec) * T(-2);
        dstd = dlogstd / std;
    }
};
// Beta with SCALAR alpha AND beta (the prior of a Beta node): the lgamma sums and the three psi values are the same for
// every element, so they are formed once per thread.  A FULL / KBCAST alpha keeps the per-element path.
template <typename T>
struct ScalarB<T, BetaOp<T>> {
    T b;
    bool hoisted;
    T lab, la_lb, psab, psa, psb;
    __device__ __forceinline__ ScalarB(T b_, T a_, bool a_scalar) : b(b_), hoisted(a_scalar) {
        if (hoisted) {
            lab = BetaOp<T>::lgab(a_, b_);
            la_lb = BetaOp<T>::lga_lgb(a_, b_);
            psab = digamma_t(a_ + b_);
            psa = digamma_t(a_);
            psb = digamma_t(b_);
        }
    }
    __device__ __forceinline__ T term(T x, T a) const {
        return hoisted ? BetaOp<T>::term_h(x, a, b, lab, la_lb) : BetaOp<T>::term(x, a, b);
    }
    template <bool NEED_X>
    __device__ __forceinline__ void grad(T g, T x, T a, T& dx, T& da, T& db) const {
        if (hoisted) BetaOp<T>::template grad_h<NEED_X>(g, x, a, b, psab, psa, psb, dx, da, db);
        else BetaOp<T>::template grad<NEED_X>(g, x, a, b, dx, da, db);
    }
};

// ---------------------------------------------------------------------------
// forward: out[r] = finish( sum_e term(x, a, b) ),  LPR lanes cooperate on a row
// ---------------------------------------------------------------------------
template <typename T, typename Op, int LPR, bool VEC>
__global__ void __launch_bounds__(256) k_rows_fwd(T* __restrict__ out, Operand<T> x, Operand<T> a, Operand<T> b,
                                                  int64_t K, int64_t M, int64_t E) {
    constexpr int VN = Pack<T>::N;
    const int lane = threadIdx.x % LPR;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    const int64_t ngrp = (int64_t)gridDim.x * blockDim.x / LPR;
    const int64_t R = K * M;
    const T xs = x.mode == ZS_SCALAR ? x.p[0] : T(0);
    const T as = a.mode == ZS_SCALAR ? a.p[0] : T(0);
    const T bs = (b.p != nullptr && b.mode == ZS_SCALAR) ? b.p[0] : T(0);
    const bool hasb = b.p != nullptr;
    const bool bsc = !hasb || b.mode == ZS_SCALAR;
    const ScalarB<T, Op> sb(bs, as, a.mode == ZS_SCALAR);

    for (int64_t base = 0; base < R; base += ngrp) {
        const int64_t r = base + grp;
        const bool valid = r < R;
        T acc = T(0);
        if (valid) {
            const int64_t m = r % M;
            const T* xr = x.row(r, m, E);
            const T* ar = a.row(r, m, E);
            const T* br = hasb ? b.row(r, m, E) : nullptr;
            if (VEC) {
                const int64_t nv = E / VN;
#pragma unroll 4
                for (int64_t v = lane; v < nv; v += LPR) {
                    Pack<T> px, pa, pb;
                    if (x.mode == ZS_SCALAR) {
#pragma unroll
                        for (int j = 0; j < VN; ++j) px.v[j] = xs;
                    } else if (x.mode == ZS_FULL) {
                        px = ld_pack_stream(xr + v * VN);
                    } else {
                        px = ld_pack(xr + v * VN);
                    }
                    if (a.mode == ZS_SCALAR) {
#pragma unroll
                        for (int j = 0; j < VN; ++j) pa.v[j] = as;
                    } else if (a.mode == ZS_FULL) {
                        pa = ld_pack_stream(ar + v * VN);
                    } else {
                        pa = ld_pack(ar + v * VN);
                    }
                    if (bsc) {
#pragma unroll
                        for (int j = 0; j < VN; ++j) acc += sb.term(px.v[j], pa.v[j]);
                    } else {
                        pb = b.mode == ZS_FULL ? ld_pack_stream(br + v * VN) : ld_pack(br + v * VN);
#pragma unroll
                        for (int j = 0; j < VN; ++j) acc += Op::term(px.v[j], pa.v[j], pb.v[j]);
                    }
                }
            } else {
                for (int64_t e = lane; e < E; e += LPR) {
                    T xv = x.mode == ZS_SCALAR ? xs : xr[e];
                    T av = a.mode == ZS_SCALAR ? as : ar[e];
                    if (bsc) acc += sb.term(xv, av);
                    else acc += Op::term(xv, av, br[e]);
                }
            }
        }
        if (LPR > 32) {
            // one CTA per row (few, long rows: the BNN likelihood [K, 1, batch]): warp sums, then a fixed-order
            // sum of the warps' partials
            __shared__ T s_part[8];
            acc = warp_sum(acc);
            __syncthreads();  // s_part may still be read from the previous row
            if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
            __syncthreads();
            acc = T(0);
#pragma unroll
            for (int w = 0; w < 8; ++w) acc += s_part[w];
        } else {
            acc = group_sum<(LPR > 32 ? 32 : LPR)>(acc);
        }
        if (valid && lane == 0) out[r] = Op::finish(acc);
    }
}

// ---------------------------------------------------------------------------
// forward for FEW, LONG rows (the BNN likelihood [K, 1, batch] of bnn_vi.py: K = 100 rows of 131 072 datapoints):
// one warp -- or one CTA -- per row leaves most of the machine idle (measured 118 GB/s, then 870 GB/s).  Here a
// thread-block CLUSTER of 8 CTAs owns a row: each CTA reduces a contiguous eighth, the partial sums meet in
// distributed shared memory (cluster.map_shared_rank) and rank 0 adds them in fixed order.  One launch, no
// workspace, deterministic.
// ---------------------------------------------------------------------------
constexpr int ROWC = 8;  // CTAs per row

template <typename T, typename Op, bool VEC>
__global__ void __cluster_dims__(ROWC, 1, 1) __launch_bounds__(256)
    k_rows_fwd_cluster(T* __restrict__ out, Operand<T> x, Operand<T> a, Operand<T> b, int64_t K, int64_t M, int64_t E) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    constexpr int VN = Pack<T>::N;
    __shared__ T s_warp[8];
    __shared__ T s_part;
    const unsigned rank = cluster.block_rank();
    const int64_t R = K * M;
    const T xs = x.mode == ZS_SCALAR ? x.p[0] : T(0);
    const T as = a.mode == ZS_SCALAR ? a.p[0] : T(0);
    const T bs = (b.p != nullptr && b.mode == ZS_SCALAR) ? b.p[0] : T(0);
    const bool hasb = b.p != nullptr;
    const bool bsc = !hasb || b.mode == ZS_SCALAR;
    const ScalarB<T, Op> sb(bs, as, a.mode == ZS_SCALAR);
    // contiguous segment of this CTA, a multiple of the pack width
    const int64_t per = ((E + (int64_t)ROWC * VN - 1) / ((int64_t)ROWC * VN)) * VN;
    const int64_t lo = (int64_t)rank * per, hi = lo + per < E ? lo + per : E;
    for (int64_t r = blockIdx.x / ROWC; r < R; r += gridDim.x / ROWC) {
        const int64_t m = r % M;
        const T* xr = x.row(r, m, E);
        const T* ar = a.row(r, m, E);
        const T* br = hasb ? b.row(r, m, E) : nullptr;
        T acc = T(0);
        if (VEC) {
#pragma unroll 4
            for (int64_t e = lo + (int64_t)threadIdx.x * VN; e < hi; e += 256 * VN) {
                Pack<T> px, pa, pb;
                if (x.mode == ZS_SCALAR) {
#pragma unroll
                    for (int j = 0; j < VN; ++j) px.v[j] = xs;
                } else {
                    px = x.mode == ZS_FULL ? ld_pack_stream(xr + e) : ld_pack(xr + e);
                }
                if (a.mode == ZS_SCALAR) {
#pragma unroll
                    for (int j = 0; j < VN; ++j) pa.v[j] = as;
                } else {
                    pa = a.mode == ZS_FULL ? ld_pack_stream(ar + e) : ld_pack(ar + e);
                }
                if (bsc) {
#pragma unroll
                    for (int j = 0; j < VN; ++j) acc += sb.term(px.v[j], pa.v[j]);
                } else {
                    pb = b.mode == ZS_FULL ? ld_pack_stream(br + e) : ld_pack(br + e);
#pragma unroll
                    for (int j = 0; j < VN; ++j) acc += Op::term(px.v[j], pa.v[j], pb.v[j]);
                }
            }
        } else {
            for (int64_t e = lo + threadIdx.x; e < hi; e += 256) {
                const T xv = x.mode == ZS_SCALAR ? xs : xr[e];
                const T av = a.mode == ZS_SCALAR ? as : ar[e];
                if (bsc) acc += sb.term(xv, av);
                else acc += Op::term(xv, av, br[e]);
            }
        }
        acc = warp_sum(acc);
        if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = acc;
        __syncthreads();
        if (threadIdx.x == 0) {
            T t = T(0);
#pragma unroll
            for (int w = 0; w < 8; ++w) t += s_warp[w];
            s_part = t;
        }
        cluster.sync();
        if (rank == 0 && threadIdx.x == 0) {
            T t = T(0);
            for (unsigned q = 0; q < ROWC; ++q) t += *cluster.map_shared_rank(&s_part, q);
            out[r] = Op::finish(t);
        }
        cluster.sync();  // partials are read before the next row overwrites them / before any CTA exits
    }
}

// ---------------------------------------------------------------------------
// backward, no reduction over K: every requested gradient has a FULL operand
// ---------------------------------------------------------------------------
template <typename T, typename Op, int LPR, bool VEC>
__global__ void __launch_bounds__(256) k_rows_bwd(T* __restrict__ dx, T* __restrict__ da, T* __restrict__ db,
                                                  const T* __restrict__ g, Operand<T> x, Operand<T> a, Operand<T> b,
                                                  int64_t K, int64_t M, int64_t E, int64_t gdiv) {
    constexpr int VN = Pack<T>::N;
    const int lane = threadIdx.x % LPR;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    const int64_t ngrp = (int64_t)gridDim.x * blockDim.x / LPR;
    const int64_t R = K * M;
    const T xs = x.mode == ZS_SCALAR ? x.p[0] : T(0);
    const T as = a.mode == ZS_SCALAR ? a.p[0] : T(0);
    const T bs = (b.p != nullptr && b.mode == ZS_SCALAR) ? b.p[0] : T(0);
    const bool hasb = b.p != nullptr;
    const bool bsc = !hasb || b.mode == ZS_SCALAR;
    const ScalarB<T, Op> sb(bs, as, a.mode == ZS_SCALAR);

    for (int64_t r = grp; r < R; r += ngrp) {
        const int64_t m = r % M;
        const T gv = g[r / gdiv];  // gdiv > 1: a long row was cut into gdiv virtual rows that share its upstream gradient
        const T* xr = x.row(r, m, E);
        const T* ar = a.row(r, m, E);
        const T* br = hasb ? b.row(r, m, E) : nullptr;
        T* dxr = dx ? dx + r * E : nullptr;
        T* dar = da ? da + r * E : nullptr;
        T* dbr = db ? db + r * E : nullptr;
        if (VEC) {
            const int64_t nv = E / VN;
#pragma unroll 2
            for (int64_t v = lane; v < nv; v += LPR) {
                Pack<T> px, pa, pb, ox, oa, ob;
                if (x.mode == ZS_SCALAR) {
#pragma unroll
                    for (int j = 0; j < VN; ++j) px.v[j] = xs;
                } else if (x.mode == ZS_FULL) {
                    px = ld_pack_stream(xr + v * VN);
                } else {
                    px = ld_pack(xr + v * VN);
                }
                if (a.mode == ZS_SCALAR) {
#pragma unroll
                    for (int j = 0; j < VN; ++j) pa.v[j] = as;
                } else if (a.mode == ZS_FULL) {
                    pa = ld_pack_stream(ar + v * VN);
                } else {
                    pa = ld_pack(ar + v * VN);
                }
                if (bsc) {
#pragma unroll
                    for (int j = 0; j < VN; ++j) {
                        if (dx) sb.template grad<true>(gv, px.v[j], pa.v[j], ox.v[j], oa.v[j], ob.v[j]);
                        else sb.template grad<false>(gv, px.v[j], pa.v[j], ox.v[j], oa.v[j], ob.v[j]);
                    }
                } else {
                    pb = b.mode == ZS_FULL ? ld_pack_stream(br + v * VN) : ld_pack(br + v * VN);
#pragma unroll
                    for (int j = 0; j < VN; ++j) {
                        if (dx)
                            Op::template grad<true>(gv, px.v[j], pa.v[j], pb.v[j], ox.v[j], oa.v[j], ob.v[j]);
                        else
                            Op::template grad<false>(gv, px.v[j], pa.v[j], pb.v[j], ox.v[j], oa.v[j], ob.v[j]);
                    }
                }
                if (dxr) st_pack_stream(dxr + v * VN, ox);
                if (dar) st_pack_stream(dar + v * VN, oa);
                if (dbr) st_pack_stream(dbr + v * VN, ob);
            }
        } else {
            for (int64_t e = lane; e < E; e += LPR) {
                T xv = x.mode == ZS_SCALAR ? xs : xr[e];
                T av = a.mode == ZS_SCALAR ? as : ar[e];
                T ox, oa, ob;
                if (bsc) {
                    if (dx) sb.template grad<true>(gv, xv, av, ox, oa, ob);
                    else sb.template grad<false>(gv, xv, av, ox, oa, ob);
                } else {
                    const T bv = br[e];
                    if (dx)
                        Op::template grad<true>(gv, xv, av, bv, ox, oa, ob);
                    else
                        Op::template grad<false>(gv, xv, av, bv, ox, oa, ob);
                }
                if (dxr) dxr[e] = ox;
                if (dar) dar[e] = oa;
                if (dbr) dbr[e] = ob;
            }
        }
    }
}

// ---------------------------------------------------------------------------
// backward with a sum over particles for KBCAST operands.
// block = (32 flat (m,e) elements) x (8 particle slices); fixed-order cross-slice sum.
// ---------------------------------------------------------------------------
constexpr int KR_X = 32, KR_Y = 8;

template <typename T, typename Op>
__global__ void __launch_bounds__(KR_X* KR_Y) k_kreduce_bwd(T* __restrict__ dx, T* __restrict__ da, T* __restrict__ db,
                                                             const T* __restrict__ g, Operand<T> x, Operand<T> a,
                                                             Operand<T> b, int64_t K, int64_t M, int64_t E) {
    const int64_t ME = M * E;
    const int64_t n = (int64_t)blockIdx.x * KR_X + threadIdx.x;
    const bool valid = n < ME;
    const int64_t m = valid ? n / E : 0;
    const bool hasb = b.p != nullptr;
    T sx = T(0), sa = T(0), sb = T(0);
    if (valid) {
        const T xs = x.mode == ZS_SCALAR ? x.p[0] : T(0);
        const T as = a.mode == ZS_SCALAR ? a.p[0] : T(0);
        const T bs = (hasb && b.mode == ZS_SCALAR) ? b.p[0] : T(0);
        const bool bsc = !hasb || b.mode == ZS_SCALAR;
        const ScalarB<T, Op> sbp(bs, as, a.mode == ZS_SCALAR);
#pragma unroll 4
        for (int64_t k = threadIdx.y; k < K; k += KR_Y) {
            const int64_t f = k * ME + n;
            T gv = g[k * M + m];
            T xv = x.mode == ZS_FULL ? x.p[f] : (x.mode == ZS_KBCAST ? x.p[n] : xs);
            T av = a.mode == ZS_FULL ? a.p[f] : (a.mode == ZS_KBCAST ? a.p[n] : as);
            T ox, oa, ob;
            if (bsc) {
                if (dx) sbp.template grad<true>(gv, xv, av, ox, oa, ob);
                else sbp.template grad<false>(gv, xv, av, ox, oa, ob);
            } else {
                const T bv = b.mode == ZS_FULL ? b.p[f] : b.p[n];
                if (dx)
                    Op::template grad<true>(gv, xv, av, bv, ox, oa, ob);
                else
                    Op::template grad<false>(gv, xv, av, bv, ox, oa, ob);
            }
            if (dx) {
                if (x.mode == ZS_FULL) dx[f] = ox; else sx += ox;
            }
            if (da) {
                if (a.mode == ZS_FULL) da[f] = oa; else sa += oa;
            }
            if (db) {
                if (b.mode == ZS_FULL) db[f] = ob; else sb += ob;
            }
        }
    }
    __shared__ T red[3][KR_Y][KR_X + 1];
    red[0][threadIdx.y][threadIdx.x] = sx;
    red[1][threadIdx.y][threadIdx.x] = sa;
    red[2][threadIdx.y][threadIdx.x] = sb;
    __syncthreads();
    if (threadIdx.y == 0 && valid) {
        T tx = T(0), ta = T(0), tb = T(0);
#pragma unroll
        for (int s = 0; s < KR_Y; ++s) {
            tx += red[0][s][threadIdx.x];
            ta += red[1][s][threadIdx.x];
            tb += red[2][s][threadIdx.x];
        }
        if (dx && x.mode == ZS_KBCAST) dx[n] = tx;
        if (da && a.mode == ZS_KBCAST) da[n] = ta;
        if (db && hasb && b.mode == ZS_KBCAST) db[n] = tb;
    }
}

// k_kreduce_bwd for the Beta op when neither parameter is FULL (the variational posterior of a Beta node: alpha and
// beta KBCAST over the K particles): psi(alpha + beta), psi(alpha) and psi(beta) depend on n only, so each thread forms
// them once, outside its particle loop, instead of once per particle.  Same block shape and fixed-order sum as
// k_kreduce_bwd; a kernel of its own so that the other ops' k_kreduce_bwd instantiations are untouched.
template <typename T>
__global__ void __launch_bounds__(KR_X* KR_Y) k_kreduce_bwd_beta(T* __restrict__ dx, T* __restrict__ da,
                                                                  T* __restrict__ db, const T* __restrict__ g,
                                                                  Operand<T> x, Operand<T> a, Operand<T> b, int64_t K,
                                                                  int64_t M, int64_t E) {
    const int64_t ME = M * E;
    const int64_t n = (int64_t)blockIdx.x * KR_X + threadIdx.x;
    const bool valid = n < ME;
    const int64_t m = valid ? n / E : 0;
    T sx = T(0), sa = T(0), sb = T(0);
    if (valid) {
        const T xs = x.mode == ZS_SCALAR ? x.p[0] : T(0);
        const T av = a.mode == ZS_KBCAST ? a.p[n] : a.p[0];
        const T bv = b.mode == ZS_KBCAST ? b.p[n] : b.p[0];
        const T psab = digamma_t(av + bv), psa = digamma_t(av), psb = digamma_t(bv);
#pragma unroll 4
        for (int64_t k = threadIdx.y; k < K; k += KR_Y) {
            const int64_t f = k * ME + n;
            const T gv = g[k * M + m];
            const T xv = x.mode == ZS_FULL ? x.p[f] : (x.mode == ZS_KBCAST ? x.p[n] : xs);
            T ox, oa, ob;
            if (dx) BetaOp<T>::template grad_h<true>(gv, xv, av, bv, psab, psa, psb, ox, oa, ob);
            else BetaOp<T>::template grad_h<false>(gv, xv, av, bv, psab, psa, psb, ox, oa, ob);
            if (dx) {
                if (x.mode == ZS_FULL) dx[f] = ox; else sx += ox;
            }
            sa += oa;
            sb += ob;
        }
    }
    __shared__ T red[3][KR_Y][KR_X + 1];
    red[0][threadIdx.y][threadIdx.x] = sx;
    red[1][threadIdx.y][threadIdx.x] = sa;
    red[2][threadIdx.y][threadIdx.x] = sb;
    __syncthreads();
    if (threadIdx.y == 0 && valid) {
        T tx = T(0), ta = T(0), tb = T(0);
#pragma unroll
        for (int s = 0; s < KR_Y; ++s) {
            tx += red[0][s][threadIdx.x];
            ta += red[1][s][threadIdx.x];
            tb += red[2][s][threadIdx.x];
        }
        if (dx && x.mode == ZS_KBCAST) dx[n] = tx;
        if (da && a.mode == ZS_KBCAST) da[n] = ta;
        if (db && b.mode == ZS_KBCAST) db[n] = tb;
    }
}

// ---------------------------------------------------------------------------
// sampling
// ---------------------------------------------------------------------------
// Normal: z = mean + std*eps over [K,N]; 4 consecutive elements per thread (one Philox call).
// Location-scale noise families: eps of  z = loc + scale * eps.
//   NOISE_NORMAL   standard normal (Box-Muller)                                        normal.py:104
//   NOISE_LOGISTIC log(u) - log(1 - u), u ~ U(0,1)                                     logistic.py:66-67
//   NOISE_LAPLACE  -sign(u) log1p(-|u|), u ~ U(-1,1)      torch.distributions.Laplace.sample (laplace.py:74)
// Injected noise (`eps_in`) is the family's UNIFORM for the last two, so the transform itself is under test.
//   NOISE_UNIFORM  u ~ U[0,1) itself                      torch.rand, as Uniform.sample draws it (uniform.py:63-66)
constexpr int NOISE_NORMAL = 0, NOISE_LOGISTIC = 1, NOISE_LAPLACE = 2, NOISE_UNIFORM = 3;

template <typename T, int NOISE>
__device__ __forceinline__ T noise_from_uniform(T u) {
    if (NOISE == NOISE_LOGISTIC) return Real<T>::log(u) - Real<T>::log(T(1) - u);
    if (NOISE == NOISE_LAPLACE) {
        const T a = u < T(0) ? -u : u;
        const T l = log1p(-a);
        return u > T(0) ? -l : (u < T(0) ? l : T(0));
    }
    return u;
}
template <int NOISE>
__device__ __forceinline__ void philox_noise4(uint64_t q, uint64_t offset, uint64_t seed, float out[4]) {
    if (NOISE == NOISE_NORMAL) {
        philox_normal4(q, offset, seed, out);
    } else {
        Philox4 r = philox4x32_10(q, offset, seed);
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (NOISE == NOISE_UNIFORM) {
                out[j] = u01_closed_open(w[j]);  // [0,1), like torch.rand
            } else {
                const float u = u01_open(w[j]);  // (0,1)
                out[j] = noise_from_uniform<float, NOISE>(NOISE == NOISE_LAPLACE ? 2.0f * u - 1.0f : u);
            }
        }
    }
}

template <typename T, bool ALIGNED4, int NOISE = NOISE_NORMAL>
__global__ void __launch_bounds__(256) k_normal_sample(T* __restrict__ z, const T* __restrict__ mean, int mm,
                                                       const T* __restrict__ std, int sm, const T* __restrict__ eps_in,
                                                       T* __restrict__ eps_out, int64_t K, int64_t N, uint64_t seed,
                                                       uint64_t offset, unsigned long long* rs,
                                                       unsigned long long* snap) {
    offset = rng_acquire(offset, rs, snap, true);
    const int64_t total = K * N;
    const int64_t nq = (total + 3) / 4;
    const T ms = mm == ZS_SCALAR ? mean[0] : T(0);
    const T ss = sm == ZS_SCALAR ? std[0] : T(0);
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        float e4[4];
        if (!eps_in) philox_noise4<NOISE>((uint64_t)q, offset, seed, e4);
        const int64_t i0 = q * 4;
        // ALIGNED4: N % 4 == 0, so the 4 elements share a particle and are contiguous in [N]
        int64_t n0 = ALIGNED4 ? (i0 % N) : 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t i = i0 + j;
            if (i < total) {
                const int64_t n = ALIGNED4 ? n0 + j : i % N;
                T e = eps_in ? noise_from_uniform<T, NOISE>(eps_in[i]) : (T)e4[j];
                T mv = mm == ZS_FULL ? mean[i] : (mm == ZS_KBCAST ? mean[n] : ms);
                T sv = sm == ZS_FULL ? std[i] : (sm == ZS_KBCAST ? std[n] : ss);
                z[i] = mv + sv * e;
                if (eps_out) eps_out[i] = e;
            }
        }
    }
}

// pathwise backward of the sample: dmean = sum_k dz ; dstd = sum_k dz*eps (KBCAST), elementwise (FULL)
template <typename T, int NOISE = NOISE_NORMAL>
__global__ void __launch_bounds__(KR_X* KR_Y) k_normal_sample_bwd(T* __restrict__ dmean, int mm, T* __restrict__ dstd,
                                                                   int sm, const T* __restrict__ dz,
                                                                   const T* __restrict__ eps, int64_t K, int64_t N,
                                                                   uint64_t seed, uint64_t offset,
                                                                   unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, false);  // the forward's snapshot: read, never advanced
    const int64_t n = (int64_t)blockIdx.x * KR_X + threadIdx.x;
    const bool valid = n < N;
    T sm_acc = T(0), ss_acc = T(0);
    if (valid) {
#pragma unroll 4
        for (int64_t k = threadIdx.y; k < K; k += KR_Y) {
            const int64_t i = k * N + n;
            T d = dz[i];
            T e;
            if (eps) {
                e = noise_from_uniform<T, NOISE>(eps[i]);
            } else {
                float e4[4];
                philox_noise4<NOISE>((uint64_t)(i >> 2), offset, seed, e4);
                e = (T)e4[i & 3];
            }
            if (dmean) {
                if (mm == ZS_FULL) dmean[i] = d; else sm_acc += d;
            }
            if (dstd) {
                if (sm == ZS_FULL) dstd[i] = d * e; else ss_acc += d * e;
            }
        }
    }
    __shared__ T red[2][KR_Y][KR_X + 1];
    red[0][threadIdx.y][threadIdx.x] = sm_acc;
    red[1][threadIdx.y][threadIdx.x] = ss_acc;
    __syncthreads();
    if (threadIdx.y == 0 && valid) {
        T tm = T(0), ts = T(0);
#pragma unroll
        for (int s = 0; s < KR_Y; ++s) {
            tm += red[0][s][threadIdx.x];
            ts += red[1][s][threadIdx.x];
        }
        if (dmean && mm == ZS_KBCAST) dmean[n] = tm;
        if (dstd && sm == ZS_KBCAST) dstd[n] = ts;
    }
}

template <typename T, bool ALIGNED4>
__global__ void __launch_bounds__(256) k_bernoulli_sample(T* __restrict__ out, const T* __restrict__ probs, int pm,
                                                          const T* __restrict__ u_in, int64_t K, int64_t N,
                                                          uint64_t seed, uint64_t offset, unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const int64_t total = K * N;
    const int64_t nq = (total + 3) / 4;
    const T ps = pm == ZS_SCALAR ? probs[0] : T(0);
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        float u4[4];
        if (!u_in) philox_uniform4((uint64_t)q, offset, seed, u4);
        const int64_t i0 = q * 4;
        int64_t n0 = ALIGNED4 ? (i0 % N) : 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t i = i0 + j;
            if (i < total) {
                const int64_t n = ALIGNED4 ? n0 + j : i % N;
                T u = u_in ? u_in[i] : (T)u4[j];
                T pv = pm == ZS_FULL ? probs[i] : (pm == ZS_KBCAST ? probs[n] : ps);
                out[i] = u < pv ? T(1) : T(0);
            }
        }
    }
}

// Poisson(rate) counts (torch.distributions.Poisson.sample as the reference calls it, zhusuan/distributions/poisson.py:61),
// drawn as ATen's CPU sample_poisson does: Knuth's product of uniforms for rate < 10, Hormann's transformed rejection
// (PTRS, "The transformed rejection method for generating Poisson random variables", 1993) for rate >= 10, in double
// for both dtypes.  Element i reads its uniforms in order from the words of Philox groups j = 0, 1, ... at counter
// i | (j << 48): a pure function of (seed, offset, i), whatever the launch geometry, and disjoint from the counters of
// the next stream position (offset + ZS_RNG_TICK).  Knuth takes one word per step, PTRS two (U, V) per trial.
// The loop stops after POISSON_MAX_WORDS words (64 groups): Knuth then returns 256, PTRS floor(rate).  For rate < 10
// Knuth needs more than 256 words only if the count exceeds 255, P < 1e-250; a PTRS trial is rejected with probability
// below 0.13 for rate >= 10, so 128 rejections in a row have P < 1e-113.  Rates are not validated (no host
// synchronisation): a negative or NaN rate gives 0, rate must be finite.
constexpr int POISSON_MAX_WORDS = 256;

struct PhiloxWords {
    uint64_t i, offset, seed;
    uint32_t w[4];
    int used;  // words consumed so far
    __device__ __forceinline__ double next() {
        if ((used & 3) == 0) {
            const Philox4 r = philox4x32_10(i | ((uint64_t)(used >> 2) << 48), offset, seed);
            w[0] = r.x; w[1] = r.y; w[2] = r.z; w[3] = r.w;
        }
        return (double)u01_closed_open(w[used++ & 3]);  // [0, 1), 24 bits
    }
};

__device__ double poisson_draw(double lam, PhiloxWords& u) {
    if (lam >= 10.0) {
        const double slam = ::sqrt(lam), loglam = ::log(lam);
        const double b = 0.931 + 2.53 * slam;
        const double a = -0.059 + 0.02483 * b;
        const double invalpha = 1.1239 + 1.1328 / (b - 3.4);
        const double vr = 0.9277 - 3.6224 / (b - 2.0);
        while (u.used < POISSON_MAX_WORDS) {
            const double U = u.next() - 0.5;
            const double V = u.next();
            const double us = 0.5 - ::fabs(U);
            const double k = ::floor((2.0 * a / us + b) * U + lam + 0.43);
            if (us >= 0.07 && V <= vr) return k;
            if (k < 0.0 || (us < 0.013 && V > us)) continue;
            if (::log(V) + ::log(invalpha) - ::log(a / (us * us) + b) <= -lam + k * loglam - ::lgamma(k + 1.0)) return k;
        }
        return ::floor(lam);
    }
    if (lam == 0.0) return 0.0;
    const double enlam = ::exp(-lam);
    double x = 0.0, prod = 1.0;
    while (u.used < POISSON_MAX_WORDS) {
        prod *= u.next();
        if (!(prod > enlam)) return x;
        x += 1.0;
    }
    return x;
}

template <typename T>
__global__ void __launch_bounds__(256) k_poisson_sample(T* __restrict__ out, const T* __restrict__ rate, int rm,
                                                        int64_t K, int64_t N, uint64_t seed, uint64_t offset,
                                                        unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const int64_t total = K * N;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const T rv = rm == ZS_FULL ? rate[i] : (rm == ZS_KBCAST ? rate[i % N] : rate[0]);
        PhiloxWords u{(uint64_t)i, offset, seed, {0u, 0u, 0u, 0u}, 0};
        out[i] = (T)poisson_draw((double)rv, u);
    }
}

// Beta(alpha, beta) samples (torch.distributions.Beta.sample, which the reference's beta.py calls), drawn as torch's
// CPU Dirichlet sampler does: G_alpha then G_beta with ATen's sample_gamma (Marsaglia and Tsang, "A simple method for
// generating gamma variables", 2000; shape < 1 boosted by (1 - u)^(1/shape) and shape + 1), each clamped below at
// DBL_MIN, and G_alpha / (G_alpha + G_beta) rounded to the output dtype and clamped to [smallest normal, nextafter(1, 0)]:
// never 0 or 1, so log_prob at a sample is finite.  Double arithmetic for both dtypes.  Element i reads its words as
// the Poisson sampler does (counter i | (j << 48)); a standard normal is Box-Muller on two words, cos branch.  A gamma
// trial takes three words (two for the normal, one uniform) and is accepted with probability above 0.95 for the boosted
// shapes >= 1; a normal with 1 + c x <= 0 is redrawn (two words).  The loop stops after BETA_MAX_WORDS words for the
// element, and a gamma draw that meets the cap returns its v = 1 point scale * d.  Meeting it takes at least 84 attempts
// with at most two acceptances among them: P < C(84, 2) 0.05^82 < 1e-100.  Parameters are not validated: alpha or beta
// that is not positive and finite (zero, negative, infinite, NaN) gives NaN.
constexpr int BETA_MAX_WORDS = 256;

__device__ __forceinline__ double philox_words_normal(PhiloxWords& u) {
    const double u1 = 1.0 - u.next();  // (0, 1]
    const double u2 = u.next();
    return ::sqrt(-2.0 * ::log(u1)) * ::cos(6.283185307179586 * u2);
}

__device__ double gamma_draw(double alpha, PhiloxWords& u) {
    double scale = 1.0;
    if (alpha < 1.0) {
        scale *= ::pow(1.0 - u.next(), 1.0 / alpha);
        alpha += 1.0;
    }
    // ATen's constants are float literals promoted to double
    const double d = alpha - (double)(1.0f / 3.0f);
    const double c = 1.0 / ::sqrt(9.0 * d);
    while (u.used < BETA_MAX_WORDS) {
        const double x = philox_words_normal(u);
        const double y = 1.0 + c * x;
        if (y <= 0.0) continue;
        const double v = y * y * y;
        const double U = 1.0 - u.next();
        const double xx = x * x;
        if (U < 1.0 - (double)0.0331f * xx * xx) return scale * d * v;
        if (::log(U) < 0.5 * xx + d * (1.0 - v + ::log(v))) return scale * d * v;
    }
    return scale * d;
}

template <typename T>
__device__ __forceinline__ T beta_clamp(double r);
template <>
__device__ __forceinline__ float beta_clamp<float>(double r) {
    return fminf(fmaxf((float)r, FLT_MIN), 0.99999994f);  // nextafterf(1, 0) = 1 - 2^-24
}
template <>
__device__ __forceinline__ double beta_clamp<double>(double r) {
    return fmin(fmax(r, DBL_MIN), 0.99999999999999989);  // nextafter(1, 0) = 1 - 2^-53
}

template <typename T>
__global__ void __launch_bounds__(256) k_beta_sample(T* __restrict__ out, const T* __restrict__ alpha, int am,
                                                     const T* __restrict__ beta, int bm, int64_t K, int64_t N,
                                                     uint64_t seed, uint64_t offset, unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const int64_t total = K * N;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const double av = (double)(am == ZS_FULL ? alpha[i] : (am == ZS_KBCAST ? alpha[i % N] : alpha[0]));
        const double bv = (double)(bm == ZS_FULL ? beta[i] : (bm == ZS_KBCAST ? beta[i % N] : beta[0]));
        if (!(av > 0.0 && bv > 0.0 && av < INFINITY && bv < INFINITY)) {
            out[i] = (T)NAN;
            continue;
        }
        PhiloxWords u{(uint64_t)i, offset, seed, {0u, 0u, 0u, 0u}, 0};
        const double ga = fmax(gamma_draw(av, u), DBL_MIN);
        const double gb = fmax(gamma_draw(bv, u), DBL_MIN);
        out[i] = beta_clamp<T>(ga / (ga + gb));
    }
}

template <typename T>
__global__ void __launch_bounds__(256) k_philox_fill(T* __restrict__ out, int64_t n, T mean, T std, int normal,
                                                     uint64_t seed, uint64_t offset, unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const int64_t nq = (n + 3) / 4;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        float v4[4];
        if (normal)
            philox_normal4((uint64_t)q, offset, seed, v4);
        else
            philox_uniform4((uint64_t)q, offset, seed, v4);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int64_t i = q * 4 + j;
            if (i < n) out[i] = normal ? mean + std * (T)v4[j] : (T)v4[j];
        }
    }
}

__global__ void __launch_bounds__(256) k_philox_raw(uint32_t* __restrict__ out, int64_t nq, uint64_t seed,
                                                    uint64_t offset, unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        Philox4 r = philox4x32_10((uint64_t)q, offset, seed);
        out[4 * q + 0] = r.x;
        out[4 * q + 1] = r.y;
        out[4 * q + 2] = r.z;
        out[4 * q + 3] = r.w;
    }
}

// ---------------------------------------------------------------------------
// host-side dispatch
// ---------------------------------------------------------------------------
// The VEC kernels walk whole packs of a row, so E % VN == 0 is needed whatever the modes are: with every operand
// SCALAR nothing else would stop a pack past E (or the dropped tail of E / VN packs).
template <typename T>
static bool vec_ok(const Operand<T>& o, int64_t E) {
    if (E % Pack<T>::N != 0) return false;
    return o.p == nullptr || o.mode == ZS_SCALAR || aligned16(o.p);
}

template <typename T, typename Op, int LPR>
static int launch_rows_fwd(T* out, Operand<T> x, Operand<T> a, Operand<T> b, int64_t K, int64_t M, int64_t E,
                           cudaStream_t st) {
    const int64_t R = K * M;
    const int rows_per_block = 256 / LPR;
    const int grid = grid_for(R, rows_per_block, 256);
    const bool vec = LPR >= 32 && vec_ok(x, E) && vec_ok(a, E) && vec_ok(b, E) && E >= Pack<T>::N;
    if (vec)
        k_rows_fwd<T, Op, LPR, true><<<grid, 256, 0, st>>>(out, x, a, b, K, M, E);
    else
        k_rows_fwd<T, Op, LPR, false><<<grid, 256, 0, st>>>(out, x, a, b, K, M, E);
    ZS_LAUNCH_CHECK("k_rows_fwd");
    return ZS_OK;
}

template <typename T, typename Op>
static int dispatch_rows_fwd(T* out, Operand<T> x, Operand<T> a, Operand<T> b, int64_t K, int64_t M, int64_t E,
                             cudaStream_t st) {
    if (K * M == 0) return ZS_OK;
    if (E <= 2) return launch_rows_fwd<T, Op, 1>(out, x, a, b, K, M, E, st);
    if (E <= 48) return launch_rows_fwd<T, Op, 8>(out, x, a, b, K, M, E, st);
    // few, long rows (one warp per row would leave most of the machine idle): one CTA per row
    if (E >= 2048 && K * M * 32 < (int64_t)sm_count() * 1024) {
        const int64_t R = K * M;
        const int64_t rows_in_flight = R < 2048 ? R : 2048;
        const bool vec = vec_ok(x, E) && vec_ok(a, E) && vec_ok(b, E);
        if (vec)
            k_rows_fwd_cluster<T, Op, true><<<(unsigned)(rows_in_flight * ROWC), 256, 0, st>>>(out, x, a, b, K, M, E);
        else
            k_rows_fwd_cluster<T, Op, false><<<(unsigned)(rows_in_flight * ROWC), 256, 0, st>>>(out, x, a, b, K, M, E);
        ZS_LAUNCH_CHECK("k_rows_fwd_cluster");
        return ZS_OK;
    }
    return launch_rows_fwd<T, Op, 32>(out, x, a, b, K, M, E, st);
}

template <typename T, typename Op, int LPR>
static int launch_rows_bwd(T* dx, T* da, T* db, const T* g, Operand<T> x, Operand<T> a, Operand<T> b, int64_t K,
                           int64_t M, int64_t E, cudaStream_t st, int64_t gdiv = 1) {
    const int64_t R = K * M;
    const int rows_per_block = 256 / LPR;
    const int grid = grid_for(R, rows_per_block, 256);
    const bool vec = LPR >= 32 && vec_ok(x, E) && vec_ok(a, E) && vec_ok(b, E) && E >= Pack<T>::N &&
                     aligned16(dx) && aligned16(da) && aligned16(db);
    if (vec)
        k_rows_bwd<T, Op, LPR, true><<<grid, 256, 0, st>>>(dx, da, db, g, x, a, b, K, M, E, gdiv);
    else
        k_rows_bwd<T, Op, LPR, false><<<grid, 256, 0, st>>>(dx, da, db, g, x, a, b, K, M, E, gdiv);
    ZS_LAUNCH_CHECK("k_rows_bwd");
    return ZS_OK;
}

template <typename T, typename Op>
static int dispatch_bwd(T* dx, T* da, T* db, const T* g, Operand<T> x, Operand<T> a, Operand<T> b, int64_t K,
                        int64_t M, int64_t E, cudaStream_t st) {
    if (K * M * E == 0) return ZS_OK;
    const bool hasb = b.p != nullptr;
    // SCALAR gradients are the host's job (it expands the operand); reject them here
    if ((dx && x.mode == ZS_SCALAR) || (da && a.mode == ZS_SCALAR) || (db && hasb && b.mode == ZS_SCALAR)) {
        set_last_error_msg("SCALAR-mode gradients are not produced by the kernels; expand the operand");
        return ZS_ERR_UNSUPPORTED;
    }
    const bool needs_kreduce =
        (dx && x.mode == ZS_KBCAST) || (da && a.mode == ZS_KBCAST) || (db && hasb && b.mode == ZS_KBCAST);
    if (needs_kreduce) {
        const int64_t ME = M * E;
        dim3 block(KR_X, KR_Y);
        const int64_t grid = (ME + KR_X - 1) / KR_X;
        ZS_REQUIRE(grid < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);
        if constexpr (std::is_same<Op, BetaOp<T>>::value) {
            if (a.mode != ZS_FULL && b.mode != ZS_FULL) {
                k_kreduce_bwd_beta<T><<<(unsigned)grid, block, 0, st>>>(dx, da, db, g, x, a, b, K, M, E);
                ZS_LAUNCH_CHECK("k_kreduce_bwd_beta");
                return ZS_OK;
            }
        }
        k_kreduce_bwd<T, Op><<<(unsigned)grid, block, 0, st>>>(dx, da, db, g, x, a, b, K, M, E);
        ZS_LAUNCH_CHECK("k_kreduce_bwd");
        return ZS_OK;
    }
    if (E <= 2) return launch_rows_bwd<T, Op, 1>(dx, da, db, g, x, a, b, K, M, E, st);
    if (E <= 48) return launch_rows_bwd<T, Op, 8>(dx, da, db, g, x, a, b, K, M, E, st);
    if (E >= 2048 && K * M * 32 < (int64_t)sm_count() * 1024) {
        // few, long rows: the backward has no reduction along the row, so a row is simply cut into S virtual rows
        // [K, M*S, E/S] (pure re-indexing for FULL and KBCAST operands alike) until the machine is full
        int64_t S = 1;
        while (S < 256 && E % (2 * S * Pack<T>::N) == 0 && E / (2 * S) >= 1024 &&
               K * M * S * 32 < (int64_t)sm_count() * 2048)
            S *= 2;
        if (S > 1) return launch_rows_bwd<T, Op, 32>(dx, da, db, g, x, a, b, K, M * S, E / S, st, S);
        return launch_rows_bwd<T, Op, 256>(dx, da, db, g, x, a, b, K, M, E, st);
    }
    return launch_rows_bwd<T, Op, 32>(dx, da, db, g, x, a, b, K, M, E, st);
}

// ---------------------------------------------------------------------------
// C-ABI entry helpers of the row log-density entry points: argument checks, dtype switch, operands.  Bernoulli, its
// logits form and Poisson have one parameter; their callers pass b = nullptr, bm = ZS_SCALAR.
// ---------------------------------------------------------------------------
template <template <typename> class Op>
constexpr bool kOneParam = false;
template <>
constexpr bool kOneParam<BernoulliOp> = true;
template <>
constexpr bool kOneParam<BernoulliLogitsOp> = true;
template <>
constexpr bool kOneParam<PoissonOp> = true;

template <template <typename> class Op>
static int rows_logprob_fwd(int dtype, void* out, const void* x, int xm, const void* a, int am, const void* b, int bm,
                            int64_t K, int64_t M, int64_t E, zs_stream_t stream) {
    ZS_REQUIRE(out && x && a && (b || kOneParam<Op>) && K >= 0 && M >= 0 && E >= 1, ZS_ERR_ARG);
    ZS_REQUIRE(valid_mode(xm) && valid_mode(am) && valid_mode(bm), ZS_ERR_ARG);
    ZS_DTYPE_SWITCH(dtype, {
        return dispatch_rows_fwd<T, Op<T>>((T*)out, Operand<T>{(const T*)x, xm}, Operand<T>{(const T*)a, am},
                                           Operand<T>{(const T*)b, bm}, K, M, E, as_stream(stream));
    })
}

template <template <typename> class Op>
static int rows_logprob_bwd(int dtype, void* dx, void* da, void* db, const void* g, const void* x, int xm,
                            const void* a, int am, const void* b, int bm, int64_t K, int64_t M, int64_t E,
                            zs_stream_t stream) {
    ZS_REQUIRE(g && x && a && (b || kOneParam<Op>) && K >= 0 && M >= 0 && E >= 1, ZS_ERR_ARG);
    ZS_REQUIRE(valid_mode(xm) && valid_mode(am) && valid_mode(bm), ZS_ERR_ARG);
    if (!dx && !da && !db) return ZS_OK;
    ZS_DTYPE_SWITCH(dtype, {
        return dispatch_bwd<T, Op<T>>((T*)dx, (T*)da, (T*)db, (const T*)g, Operand<T>{(const T*)x, xm},
                                      Operand<T>{(const T*)a, am}, Operand<T>{(const T*)b, bm}, K, M, E,
                                      as_stream(stream));
    })
}

// f(OpTag<Op>{}) with the per-element Op of a zs_locscale_logprob_* family; ZS_ERR_ARG for an unknown family
template <template <typename> class FamilyOp>
struct OpTag {
    template <typename T>
    using Op = FamilyOp<T>;
};
template <typename F>
static int with_locscale_op(int family, F&& f) {
    switch (family) {
        case ZS_FAM_LOGISTIC: return f(OpTag<LogisticOp>{});
        case ZS_FAM_LAPLACE: return f(OpTag<LaplaceOp>{});
        case ZS_FAM_UNIFORM: return f(OpTag<UniformOp>{});  // loc = low, scale = high
        case ZS_FAM_BETA: return f(OpTag<BetaOp>{});        // loc = alpha, scale = beta
    }
    set_last_error_msg("family must be ZS_FAM_LOGISTIC, ZS_FAM_LAPLACE, ZS_FAM_UNIFORM or ZS_FAM_BETA");
    return ZS_ERR_ARG;
}

// f(integral_constant<int, NOISE_*>{}) with the sampler noise of a zs_locscale_sample* family; ZS_ERR_ARG for any other
template <typename F>
static int with_locscale_noise(int family, F&& f) {
    switch (family) {
        case ZS_FAM_LOGISTIC: return f(std::integral_constant<int, NOISE_LOGISTIC>{});
        case ZS_FAM_LAPLACE: return f(std::integral_constant<int, NOISE_LAPLACE>{});
        case ZS_FAM_UNIFORM: return f(std::integral_constant<int, NOISE_UNIFORM>{});
    }
    set_last_error_msg("family must be ZS_FAM_LOGISTIC, ZS_FAM_LAPLACE or ZS_FAM_UNIFORM");
    return ZS_ERR_ARG;
}

}  // namespace zs

using namespace zs;

__global__ void k_rng_state_init(unsigned long long* st, unsigned long long offset) {
    st[0] = offset;
    st[1] = 0ull;
}
static inline unsigned long long* rs_ptr(const void* p) {
    return reinterpret_cast<unsigned long long*>(const_cast<void*>(p));
}

extern "C" {

int zs_rng_state_init(void* rng_state, uint64_t offset, zs_stream_t stream) {
    ZS_REQUIRE(rng_state != nullptr && (reinterpret_cast<uintptr_t>(rng_state) & 7u) == 0, ZS_ERR_ARG);
    k_rng_state_init<<<1, 1, 0, as_stream(stream)>>>((unsigned long long*)rng_state, offset);
    ZS_LAUNCH_CHECK("k_rng_state_init");
    return ZS_OK;
}

int zs_philox_raw(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(out != nullptr && n >= 0 && n % 4 == 0, ZS_ERR_ARG);
    if (n == 0) return ZS_OK;
    k_philox_raw<<<grid_for(n / 4, 256), 256, 0, as_stream(stream)>>>(out, n / 4, seed, offset, rs_ptr(rng_state));
    ZS_LAUNCH_CHECK("k_philox_raw");
    return ZS_OK;
}

int zs_philox_uniform(int dtype, void* out, int64_t n, uint64_t seed, uint64_t offset, void* rng_state,
                      zs_stream_t stream) {
    ZS_REQUIRE(out != nullptr && n >= 0, ZS_ERR_ARG);
    if (n == 0) return ZS_OK;
    ZS_DTYPE_SWITCH(dtype, {
        k_philox_fill<T><<<grid_for((n + 3) / 4, 256), 256, 0, as_stream(stream)>>>((T*)out, n, T(0), T(1), 0, seed,
                                                                                     offset, rs_ptr(rng_state));
    })
    ZS_LAUNCH_CHECK("k_philox_fill");
    return ZS_OK;
}

int zs_philox_normal(int dtype, void* out, int64_t n, double mean, double std, uint64_t seed, uint64_t offset,
                     void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(out != nullptr && n >= 0, ZS_ERR_ARG);
    if (n == 0) return ZS_OK;
    ZS_DTYPE_SWITCH(dtype, {
        k_philox_fill<T><<<grid_for((n + 3) / 4, 256), 256, 0, as_stream(stream)>>>((T*)out, n, (T)mean, (T)std, 1,
                                                                                     seed, offset, rs_ptr(rng_state));
    })
    ZS_LAUNCH_CHECK("k_philox_fill");
    return ZS_OK;
}

int zs_normal_sample(int dtype, void* z, const void* mean, int mean_mode, const void* std, int std_mode,
                     const void* eps_in, void* eps_out, int64_t K, int64_t N, uint64_t seed, uint64_t offset,
                     void* rng_state, void* rng_snapshot, zs_stream_t stream) {
    ZS_REQUIRE(z && mean && std && K >= 0 && N >= 0, ZS_ERR_ARG);
    if (eps_in) rng_state = rng_snapshot = nullptr;  // injected noise: no draw, the stream position stays
    ZS_REQUIRE(valid_mode(mean_mode) && valid_mode(std_mode), ZS_ERR_ARG);
    if (K * N == 0) return ZS_OK;
    const int grid = grid_for((K * N + 3) / 4, 256);
    ZS_DTYPE_SWITCH(dtype, {
        if (N % 4 == 0)
            k_normal_sample<T, true><<<grid, 256, 0, as_stream(stream)>>>(
                (T*)z, (const T*)mean, mean_mode, (const T*)std, std_mode, (const T*)eps_in, (T*)eps_out, K, N, seed,
                offset, rs_ptr(rng_state), rs_ptr(rng_snapshot));
        else
            k_normal_sample<T, false><<<grid, 256, 0, as_stream(stream)>>>(
                (T*)z, (const T*)mean, mean_mode, (const T*)std, std_mode, (const T*)eps_in, (T*)eps_out, K, N, seed,
                offset, rs_ptr(rng_state), rs_ptr(rng_snapshot));
    })
    ZS_LAUNCH_CHECK("k_normal_sample");
    return ZS_OK;
}

int zs_normal_sample_bwd(int dtype, void* dmean, int mean_mode, void* dstd, int std_mode, const void* dz,
                         const void* eps, int64_t K, int64_t N, uint64_t seed, uint64_t offset, const void* rng_state,
                         zs_stream_t stream) {
    ZS_REQUIRE(dz && K >= 0 && N >= 0, ZS_ERR_ARG);
    ZS_REQUIRE(valid_mode(mean_mode) && valid_mode(std_mode), ZS_ERR_ARG);
    if ((dmean && mean_mode == ZS_SCALAR) || (dstd && std_mode == ZS_SCALAR)) {
        set_last_error_msg("SCALAR-mode gradients are not produced by the kernels; expand the operand");
        return ZS_ERR_UNSUPPORTED;
    }
    if (K * N == 0 || (!dmean && !dstd)) return ZS_OK;
    dim3 block(KR_X, KR_Y);
    const int64_t grid = (N + KR_X - 1) / KR_X;
    ZS_REQUIRE(grid < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);
    ZS_DTYPE_SWITCH(dtype, {
        k_normal_sample_bwd<T><<<(unsigned)grid, block, 0, as_stream(stream)>>>(
            (T*)dmean, mean_mode, (T*)dstd, std_mode, (const T*)dz, (const T*)eps, K, N, seed, offset,
            eps ? nullptr : rs_ptr(rng_state));
    })
    ZS_LAUNCH_CHECK("k_normal_sample_bwd");
    return ZS_OK;
}

int zs_normal_logprob_fwd(int dtype, void* out, const void* x, int x_mode, const void* mean, int mean_mode,
                          const void* std, int std_mode, int64_t K, int64_t M, int64_t E, zs_stream_t stream) {
    return rows_logprob_fwd<NormalOp>(dtype, out, x, x_mode, mean, mean_mode, std, std_mode, K, M, E, stream);
}

int zs_normal_logprob_bwd(int dtype, void* dx, void* dmean, void* dstd, const void* g, const void* x, int x_mode,
                          const void* mean, int mean_mode, const void* std, int std_mode, int64_t K, int64_t M,
                          int64_t E, zs_stream_t stream) {
    return rows_logprob_bwd<NormalOp>(dtype, dx, dmean, dstd, g, x, x_mode, mean, mean_mode, std, std_mode, K, M, E,
                                      stream);
}

int zs_bernoulli_sample(int dtype, void* out, const void* probs, int probs_mode, const void* u_in, int64_t K,
                        int64_t N, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(out && probs && K >= 0 && N >= 0 && valid_mode(probs_mode), ZS_ERR_ARG);
    if (u_in) rng_state = nullptr;
    if (K * N == 0) return ZS_OK;
    const int grid = grid_for((K * N + 3) / 4, 256);
    ZS_DTYPE_SWITCH(dtype, {
        if (N % 4 == 0)
            k_bernoulli_sample<T, true><<<grid, 256, 0, as_stream(stream)>>>((T*)out, (const T*)probs, probs_mode,
                                                                              (const T*)u_in, K, N, seed, offset,
                                                                              rs_ptr(rng_state));
        else
            k_bernoulli_sample<T, false><<<grid, 256, 0, as_stream(stream)>>>((T*)out, (const T*)probs, probs_mode,
                                                                               (const T*)u_in, K, N, seed, offset,
                                                                               rs_ptr(rng_state));
    })
    ZS_LAUNCH_CHECK("k_bernoulli_sample");
    return ZS_OK;
}

int zs_bernoulli_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* probs, int probs_mode,
                            int64_t K, int64_t M, int64_t E, zs_stream_t stream) {
    return rows_logprob_fwd<BernoulliOp>(dtype, out, x, x_mode, probs, probs_mode, nullptr, ZS_SCALAR, K, M, E, stream);
}

int zs_bernoulli_logpmf_bwd(int dtype, void* dx, void* dprobs, const void* g, const void* x, int x_mode,
                            const void* probs, int probs_mode, int64_t K, int64_t M, int64_t E, zs_stream_t stream) {
    return rows_logprob_bwd<BernoulliOp>(dtype, dx, dprobs, nullptr, g, x, x_mode, probs, probs_mode, nullptr,
                                         ZS_SCALAR, K, M, E, stream);
}

/* ---- location-scale families beyond Normal (SURVEY 8(f)-4) ------------------------------------------------ */
int zs_locscale_sample(int dtype, int family, void* z, const void* loc, int loc_mode, const void* scale, int scale_mode,
                       const void* u_in, int64_t K, int64_t N, uint64_t seed, uint64_t offset, void* rng_state,
                       void* rng_snapshot, zs_stream_t stream) {
    ZS_REQUIRE(z && loc && scale && K >= 0 && N >= 0, ZS_ERR_ARG);
    if (u_in) rng_state = rng_snapshot = nullptr;
    ZS_REQUIRE(valid_mode(loc_mode) && valid_mode(scale_mode), ZS_ERR_ARG);
    return with_locscale_noise(family, [&](auto noise) -> int {
        if (K * N == 0) return ZS_OK;
        const int grid = grid_for((K * N + 3) / 4, 256);
        ZS_DTYPE_SWITCH(dtype, {
            k_normal_sample<T, false, decltype(noise)::value><<<grid, 256, 0, as_stream(stream)>>>(
                (T*)z, (const T*)loc, loc_mode, (const T*)scale, scale_mode, (const T*)u_in, (T*)nullptr, K, N, seed,
                offset, rs_ptr(rng_state), rs_ptr(rng_snapshot));
        })
        ZS_LAUNCH_CHECK("k_normal_sample<locscale>");
        return ZS_OK;
    });
}

int zs_locscale_sample_bwd(int dtype, int family, void* dloc, int loc_mode, void* dscale, int scale_mode, const void* dz,
                           const void* u, int64_t K, int64_t N, uint64_t seed, uint64_t offset, const void* rng_state,
                           zs_stream_t stream) {
    ZS_REQUIRE(dz && K >= 0 && N >= 0, ZS_ERR_ARG);
    ZS_REQUIRE(valid_mode(loc_mode) && valid_mode(scale_mode), ZS_ERR_ARG);
    return with_locscale_noise(family, [&](auto noise) -> int {
        if ((dloc && loc_mode == ZS_SCALAR) || (dscale && scale_mode == ZS_SCALAR)) {
            set_last_error_msg("SCALAR-mode gradients are not produced by the kernels; expand the operand");
            return ZS_ERR_UNSUPPORTED;
        }
        if (K * N == 0 || (!dloc && !dscale)) return ZS_OK;
        dim3 block(KR_X, KR_Y);
        const int64_t grid = (N + KR_X - 1) / KR_X;
        ZS_REQUIRE(grid < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);
        ZS_DTYPE_SWITCH(dtype, {
            k_normal_sample_bwd<T, decltype(noise)::value><<<(unsigned)grid, block, 0, as_stream(stream)>>>(
                (T*)dloc, loc_mode, (T*)dscale, scale_mode, (const T*)dz, (const T*)u, K, N, seed, offset,
                u ? nullptr : rs_ptr(rng_state));
        })
        ZS_LAUNCH_CHECK("k_normal_sample_bwd<locscale>");
        return ZS_OK;
    });
}

int zs_locscale_logprob_fwd(int dtype, int family, void* out, const void* x, int x_mode, const void* loc, int loc_mode,
                            const void* scale, int scale_mode, int64_t K, int64_t M, int64_t E, zs_stream_t stream) {
    return with_locscale_op(family, [&](auto tag) {
        return rows_logprob_fwd<decltype(tag)::template Op>(dtype, out, x, x_mode, loc, loc_mode, scale, scale_mode, K,
                                                            M, E, stream);
    });
}

int zs_locscale_logprob_bwd(int dtype, int family, void* dx, void* dloc, void* dscale, const void* g, const void* x,
                            int x_mode, const void* loc, int loc_mode, const void* scale, int scale_mode, int64_t K,
                            int64_t M, int64_t E, zs_stream_t stream) {
    return with_locscale_op(family, [&](auto tag) {
        return rows_logprob_bwd<decltype(tag)::template Op>(dtype, dx, dloc, dscale, g, x, x_mode, loc, loc_mode, scale,
                                                            scale_mode, K, M, E, stream);
    });
}

int zs_bernoulli_logits_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* logits, int logits_mode,
                                   int64_t K, int64_t M, int64_t E, zs_stream_t stream) {
    return rows_logprob_fwd<BernoulliLogitsOp>(dtype, out, x, x_mode, logits, logits_mode, nullptr, ZS_SCALAR, K, M, E,
                                               stream);
}

int zs_bernoulli_logits_logpmf_bwd(int dtype, void* dx, void* dlogits, const void* g, const void* x, int x_mode,
                                   const void* logits, int logits_mode, int64_t K, int64_t M, int64_t E,
                                   zs_stream_t stream) {
    return rows_logprob_bwd<BernoulliLogitsOp>(dtype, dx, dlogits, nullptr, g, x, x_mode, logits, logits_mode, nullptr,
                                               ZS_SCALAR, K, M, E, stream);
}

/* ---- Poisson stochastic node ---------------------------------------------------------------------------- */
int zs_poisson_sample(int dtype, void* out, const void* rate, int rate_mode, int64_t K, int64_t N, uint64_t seed,
                      uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(out && rate && K >= 0 && N >= 0 && valid_mode(rate_mode), ZS_ERR_ARG);
    if (K * N == 0) return ZS_OK;
    ZS_REQUIRE(K * N < ((int64_t)1 << 48), ZS_ERR_UNSUPPORTED);  // element index below the group bits of the counter
    const int grid = grid_for(K * N, 256);
    ZS_DTYPE_SWITCH(dtype, {
        k_poisson_sample<T><<<grid, 256, 0, as_stream(stream)>>>((T*)out, (const T*)rate, rate_mode, K, N, seed, offset,
                                                                 rs_ptr(rng_state));
    })
    ZS_LAUNCH_CHECK("k_poisson_sample");
    return ZS_OK;
}

int zs_poisson_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* rate, int rate_mode, int64_t K,
                          int64_t M, int64_t E, zs_stream_t stream) {
    return rows_logprob_fwd<PoissonOp>(dtype, out, x, x_mode, rate, rate_mode, nullptr, ZS_SCALAR, K, M, E, stream);
}

int zs_poisson_logpmf_bwd(int dtype, void* drate, const void* g, const void* x, int x_mode, const void* rate,
                          int rate_mode, int64_t K, int64_t M, int64_t E, zs_stream_t stream) {
    return rows_logprob_bwd<PoissonOp>(dtype, nullptr, drate, nullptr, g, x, x_mode, rate, rate_mode, nullptr, ZS_SCALAR,
                                       K, M, E, stream);
}

/* ---- Beta stochastic node (log-density: zs_locscale_logprob_* with ZS_FAM_BETA) ------------------------------ */
int zs_beta_sample(int dtype, void* out, const void* alpha, int alpha_mode, const void* beta, int beta_mode, int64_t K,
                   int64_t N, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(out && alpha && beta && K >= 0 && N >= 0 && valid_mode(alpha_mode) && valid_mode(beta_mode), ZS_ERR_ARG);
    if (K * N == 0) return ZS_OK;
    ZS_REQUIRE(K * N < ((int64_t)1 << 48), ZS_ERR_UNSUPPORTED);  // element index below the group bits of the counter
    const int grid = grid_for(K * N, 256);
    ZS_DTYPE_SWITCH(dtype, {
        k_beta_sample<T><<<grid, 256, 0, as_stream(stream)>>>((T*)out, (const T*)alpha, alpha_mode, (const T*)beta,
                                                              beta_mode, K, N, seed, offset, rs_ptr(rng_state));
    })
    ZS_LAUNCH_CHECK("k_beta_sample");
    return ZS_OK;
}

}  // extern "C"
