// Multi-particle objectives over log-weights [K,B], forward + backward in one launch.
//
// Replaces (reference file:line):
//   compute_iw_term                      zhusuan/variational/importance_weighted_objective.py:16-25
//   ImportanceWeightedObjective.sgvb     zhusuan/variational/importance_weighted_objective.py:102-132
//   ImportanceWeightedObjective.vimco    zhusuan/variational/importance_weighted_objective.py:134-191
//   log_mean_exp                         zhusuan/utils.py:6-21
// The reference materialises a [B,K,K] tensor for the VIMCO leave-one-out baseline (:184-186) and
// runs ~40 aten kernels; here each batch column is reduced over its K particles with O(K) work:
//   x_k = logp_k - logq_k, m = max x, e_k = exp(x_k - m), S = sum e, wt_k = e_k / S
//   sgvb : cost = -sum wt_k x_k ;              dlogp = -wt,  dlogq = +wt
//   vimco: mu_k = (sum_j x_j - x_k)/(K-1)      (log geometric mean of the other weights)
//          sig_k = L - loo_k = -log1p( (exp(mu_k - m) - e_k) / S )
//          cost = -sum logq_k sig_k - sum wt_k x_k ;  dlogp = -wt, dlogq = wt - sig
// sig is formed without the reference's L - loo cancellation, so it is at least as accurate as the
// reference's fp32 result (DESIGN.md §numerics).
#include "zs_common.cuh"

#include <cooperative_groups.h>

namespace zs {

constexpr int OBJ_THREADS = 256;

// deterministic reduction across the k-slices (threadIdx.y) of one column (threadIdx.x)
template <typename T, typename F>
__device__ __forceinline__ T slice_reduce(T v, T* sm, int cols, int slices, F f) {
    sm[threadIdx.y * cols + threadIdx.x] = v;
    __syncthreads();
    // tree over slices, fixed order
    for (int s = 1; s < slices; s <<= 1) {
        if ((threadIdx.y % (2 * s)) == 0 && threadIdx.y + s < slices)
            sm[threadIdx.y * cols + threadIdx.x] =
                f(sm[threadIdx.y * cols + threadIdx.x], sm[(threadIdx.y + s) * cols + threadIdx.x]);
        __syncthreads();
    }
    T r = sm[threadIdx.x];
    __syncthreads();
    return r;
}

template <typename T>
struct Top2 {
    T m1, m2;
    long long i1;
};

// Log-weights are formed and centred in double: |log w| is O(100-1000), where fp32 has an ulp of
// ~6e-5 that exp() would turn into ~1e-4 relative noise on every weight (the reference's own fp32
// noise floor, SURVEY.md §8c).  Only the small centred difference is rounded to T before exp().
template <typename T, int EST>
__global__ void __launch_bounds__(OBJ_THREADS)
    k_iw_objective(T* __restrict__ cost, T* __restrict__ dlogp, T* __restrict__ dlogq, const T* __restrict__ logp,
                   const T* __restrict__ logq, const T* __restrict__ extra, int64_t K, int64_t B, T gscale, int cols,
                   int slices) {
    using A = double;
    extern __shared__ unsigned char smem_raw[];
    A* sm = reinterpret_cast<A*>(smem_raw);                           // [slices*cols]
    long long* smi = reinterpret_cast<long long*>(sm + OBJ_THREADS);  // [slices*cols]
    const int64_t b = (int64_t)blockIdx.x * cols + threadIdx.x;
    const bool valid = b < B;
    const A NEG_INF = -INFINITY;
    auto logw = [&](int64_t k) -> A {
        return ((A)logp[k * B + b] - (A)logq[k * B + b]) + (extra ? (A)extra[k * B + b] : A(0));
    };

    if (EST == ZS_EST_ELBO) {
        // ELBO.sgvb (elbo.py:155-156): -mean over particles of (logp - logq); d/dlogp = -1/K, d/dlogq = +1/K
        A acc = A(0);
        const T gk = gscale / (T)K;
        if (valid) {
            for (int64_t k = threadIdx.y; k < K; k += slices) {
                acc -= logw(k);
                if (dlogp) dlogp[k * B + b] = -gk;
                if (dlogq) dlogq[k * B + b] = gk;
            }
        }
        acc = slice_reduce(acc, sm, cols, slices, [](A a, A c) { return a + c; });
        if (valid && threadIdx.y == 0 && cost) cost[b] = (T)(acc / (A)K);
        return;
    }

    // pass 1: max (and, for VIMCO, second max excluding the first argmax)
    A m1 = NEG_INF, m2 = NEG_INF, sumd = A(0);
    long long i1 = -1;
    if (valid) {
        for (int64_t k = threadIdx.y; k < K; k += slices) {
            A x = logw(k);
            if (x > m1 || i1 < 0) {
                m2 = m1;
                m1 = x;
                i1 = k;
            } else if (x > m2) {
                m2 = x;
            }
        }
    }
    // merge (m1,i1,m2) across slices: smallest index wins ties so the result is order independent
    {
        sm[threadIdx.y * cols + threadIdx.x] = m1;
        smi[threadIdx.y * cols + threadIdx.x] = i1;
        __syncthreads();
        A gm = NEG_INF;
        long long gi = -1;
        for (int s = 0; s < slices; ++s) {
            A v = sm[s * cols + threadIdx.x];
            long long vi = smi[s * cols + threadIdx.x];
            if (vi >= 0 && (gi < 0 || v > gm || (v == gm && vi < gi))) {
                gm = v;
                gi = vi;
            }
        }
        __syncthreads();
        if (EST == ZS_EST_VIMCO) {
            // second max = max over all elements except index gi
            A cand = (i1 == gi) ? m2 : m1;
            m2 = slice_reduce(cand, sm, cols, slices, [](A a, A c) { return a > c ? a : c; });
        }
        m1 = gm;
        i1 = gi;
    }
    const T gap = (T)(m1 - m2);

    // pass 2: S = sum exp(x - m) ; VIMCO also S2 = sum_{k != argmax} exp(x - m2) and sum (x - m):
    // the leave-one-out mean is only ever needed relative to m, and summing the centred values
    // keeps its rounding error ~|spread|*eps instead of ~K*|log w|*eps
    A S_a = A(0), S2_a = A(0);
    if (valid) {
        for (int64_t k = threadIdx.y; k < K; k += slices) {
            A x = logw(k);
            S_a += (A)Real<T>::exp((T)(x - m1));
            if (EST == ZS_EST_VIMCO) {
                sumd += x - m1;
                if (k != i1) S2_a += (A)Real<T>::exp((T)(x - m2));
            }
        }
    }
    const T S = (T)slice_reduce(S_a, sm, cols, slices, [](A a, A c) { return a + c; });
    T S2 = T(0);
    if (EST == ZS_EST_VIMCO) {
        S2 = (T)slice_reduce(S2_a, sm, cols, slices, [](A a, A c) { return a + c; });
        sumd = slice_reduce(sumd, sm, cols, slices, [](A a, A c) { return a + c; });
    }

    // pass 3: weights, learning signal, cost and gradients
    A c_acc = A(0);
    if (valid) {
        const T invS = T(1) / S;
        const A km1 = (A)(K - 1);
        for (int64_t k = threadIdx.y; k < K; k += slices) {
            const T lq = logq[k * B + b];
            const A x = logw(k);
            const T e = Real<T>::exp((T)(x - m1));
            const T wt = e / S;
            c_acc -= (A)wt * x;
            T gq = wt;
            if (EST == ZS_EST_VIMCO) {
                const T mu_m = (T)((sumd - (x - m1)) / km1);  // LOO mean of log w, minus m
                T sig;
                if (k == i1 && gap > T(1)) {
                    // the arg-max row: S - e would cancel, re-centre on the second max
                    T Sloo = S2 + Real<T>::exp(mu_m + gap);
                    sig = gap + (Real<T>::log(S) - Real<T>::log(Sloo));
                } else {
                    T t = (Real<T>::exp(mu_m) - e) * invS;
                    sig = -log1p(t);
                }
                c_acc -= (A)lq * (A)sig;
                gq = wt - sig;
            }
            if (dlogp) dlogp[k * B + b] = -wt * gscale;
            if (dlogq) dlogq[k * B + b] = gq * gscale;
        }
    }
    c_acc = slice_reduce(c_acc, sm, cols, slices, [](A a, A c) { return a + c; });
    if (valid && threadIdx.y == 0 && cost) cost[b] = (T)c_acc;
}

template <typename T, bool BWD>
__global__ void __launch_bounds__(OBJ_THREADS)
    k_log_mean_exp(T* __restrict__ out, const T* __restrict__ g, const T* __restrict__ x, int64_t K, int64_t B,
                   int cols, int slices) {
    extern __shared__ unsigned char smem_raw[];
    T* sm = reinterpret_cast<T*>(smem_raw);
    const int64_t b = (int64_t)blockIdx.x * cols + threadIdx.x;
    const bool valid = b < B;
    T m = -INFINITY;
    if (valid)
        for (int64_t k = threadIdx.y; k < K; k += slices) m = fmax(m, x[k * B + b]);
    m = slice_reduce(m, sm, cols, slices, [](T a, T c) { return a > c ? a : c; });
    T S = T(0);
    if (valid)
        for (int64_t k = threadIdx.y; k < K; k += slices) S += Real<T>::exp(x[k * B + b] - m);
    S = slice_reduce(S, sm, cols, slices, [](T a, T c) { return a + c; });
    if (!BWD) {
        // zhusuan/utils.py:18-19: log(mean(exp(x - max))) + max
        if (valid && threadIdx.y == 0) out[b] = Real<T>::log(S / (T)K) + m;
    } else if (valid) {
        const T gb = g[b];
        for (int64_t k = threadIdx.y; k < K; k += slices) out[k * B + b] = gb * (Real<T>::exp(x[k * B + b] - m) / S);
    }
}

// buf *= *scale, skipped entirely when *scale == 1 (the usual loss.backward() case): lets a fused
// forward+backward kernel hand out gradients computed for a unit upstream gradient without a host
// sync and without a second pass over them.
template <typename T>
__device__ __forceinline__ void scale_buffer(T* __restrict__ buf, int64_t n, T s) {
    if (buf == nullptr) return;
    constexpr int VN = Pack<T>::N;
    const int64_t nv = n / VN;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nv; v += stride) {
        Pack<T> p = ld_pack(buf + v * VN);
#pragma unroll
        for (int j = 0; j < VN; ++j) p.v[j] *= s;
        st_pack(buf + v * VN, p);
    }
    for (int64_t i = nv * VN + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) buf[i] *= s;
}
// up to three buffers (the fused objective's dprobs, dlogp, dlogq) in one launch
template <typename T>
__global__ void __launch_bounds__(256) k_scale_inplace(T* __restrict__ b0, int64_t n0, T* __restrict__ b1, int64_t n1,
                                                       T* __restrict__ b2, int64_t n2, const T* __restrict__ scale) {
    pdl_wait();
    pdl_trigger();
    const T s = *scale;
    if (s == T(1)) return;
    scale_buffer(b0, n0, s);
    scale_buffer(b1, n1, s);
    scale_buffer(b2, n2, s);
}

static void column_geometry(int64_t B, int& cols, int& slices) {
    cols = 1;
    while (cols < 32 && cols < B) cols <<= 1;
    slices = OBJ_THREADS / cols;
}

// ---------------------------------------------------------------------------------------------
// ELBO.reinforce (zhusuan/variational/elbo.py:163-238), the common form: variance reduction with the moving-mean
// baseline, no user baseline, mean over all axes.  The reference runs ~15 aten kernels and keeps the state on the
// host; here ONE launch of ONE thread-block cluster (8 CTAs, distributed shared memory) does
//   s_i = logp_i - logq_i ;  bc = mean_i s_i                                      (:206-219)
//   mm <- mm - (mm - bc)(1 - decay) ; step <- step + 1 ; mm <- mm / (1 - decay^step)   (:221-224, float32 state,
//                                                                             bias-corrected IN PLACE as the reference)
//   sig_i = s_i - mm ;  cost = -mean_i( logp_i + sig_i logq_i )                   (:225-238)
//   dlogp_i = -gscale ;  dlogq_i = -sig_i gscale                                  (autograd of the surrogate)
// The [N] arrays are small ([K,B], 0.2 MB at config 2): the kernel is latency-bound by design, the cluster only
// keeps the two passes and both reductions inside one launch.  Reductions are fixed-order (deterministic).
// ---------------------------------------------------------------------------------------------
constexpr int RF_CLUSTER = 8;
constexpr int RF_THREADS = 512;

__device__ __forceinline__ double rf_block_sum(double v, double* s_warp) {
    v = warp_sum(v);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    __syncthreads();  // s_warp may still be read from the previous reduction
    if (lane == 0) s_warp[warp] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < RF_THREADS / 32; ++w) t += s_warp[w];  // fixed order, every thread
    return t;
}

template <typename T>
__global__ void __cluster_dims__(RF_CLUSTER, 1, 1) __launch_bounds__(RF_THREADS)
    k_reinforce(T* __restrict__ cost, T* __restrict__ dlogp, T* __restrict__ dlogq, float* __restrict__ moving_mean,
                int* __restrict__ local_step, const T* __restrict__ logp, const T* __restrict__ logq, int64_t N,
                float decay, T gscale) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double s_warp[RF_THREADS / 32];
    __shared__ double s_part[2];  // [0]: sum of s over this CTA's slice, [1]: sum of the surrogate terms
    const unsigned rank = cluster.block_rank();
    const int64_t per = (N + RF_CLUSTER - 1) / RF_CLUSTER;
    const int64_t lo = (int64_t)rank * per, hi = (lo + per < N) ? lo + per : N;
    // the state is read by every CTA before CTA 0 overwrites it (ordered by the first cluster barrier)
    const float mm_old = *moving_mean;
    const int step = *local_step + 1;

    double acc = 0.0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += RF_THREADS) acc += (double)logp[i] - (double)logq[i];
    acc = rf_block_sum(acc, s_warp);
    if (threadIdx.x == 0) s_part[0] = acc;
    cluster.sync();
    double total = 0.0;
    for (unsigned r = 0; r < RF_CLUSTER; ++r) total += *cluster.map_shared_rank(&s_part[0], r);
    const T bc = (T)(total / (double)N);
    // float32 state arithmetic, in the reference's operation order
    float mm;
    if (sizeof(T) == 4) mm = mm_old - (mm_old - (float)bc) * (float)(1.0 - (double)decay);
    else mm = (float)((double)mm_old - ((double)mm_old - (double)bc) * (1.0 - (double)decay));
    const float bias = 1.0f - powf(decay, (float)step);
    mm = mm / bias;
    if (rank == 0 && threadIdx.x == 0) {
        *moving_mean = mm;
        *local_step = step;
    }

    double cacc = 0.0;
    for (int64_t i = lo + threadIdx.x; i < hi; i += RF_THREADS) {
        const T lp = logp[i], lq = logq[i];
        const T sig = (lp - lq) - (T)mm;
        cacc += (double)(lp + sig * lq);
        if (dlogp) dlogp[i] = -gscale;
        if (dlogq) dlogq[i] = -sig * gscale;
    }
    cacc = rf_block_sum(cacc, s_warp);
    if (threadIdx.x == 0) s_part[1] = cacc;
    cluster.sync();
    if (rank == 0 && threadIdx.x == 0) {
        double c = 0.0;
        for (unsigned r = 0; r < RF_CLUSTER; ++r) c += *cluster.map_shared_rank(&s_part[1], r);
        *cost = (T)(-(c / (double)N));
    }
    cluster.sync();  // no CTA may exit while CTA 0 still reads its shared memory
}

// ---------------------------------------------------------------------------------------------
// out[0] = sa * sum(a) + sb * sum(b): the scalar that ELBO.sgvb returns when a flow is attached
// (zhusuan/variational/elbo.py:155-161: -mean(logp - logq) - sum(log_det)) from the per-column costs and the flow's
// log-determinants, in ONE launch with a fixed summation order (thread t adds elements t, t + 1024, ...; the partials are
// combined by a shuffle tree and a fixed loop over the warps) instead of a mean, a sum and a subtraction kernel.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(1024) k_combine_sums(T* __restrict__ out, const T* __restrict__ a, int64_t na, T sa,
                                                       const T* __restrict__ b, int64_t nb, T sb) {
    double acc_a = 0.0, acc_b = 0.0;
    for (int64_t i = threadIdx.x; i < na; i += 1024) acc_a += (double)a[i];
    for (int64_t i = threadIdx.x; i < nb; i += 1024) acc_b += (double)b[i];
    double v = (double)sa * acc_a + (double)sb * acc_b;
    v = warp_sum(v);
    __shared__ double s_part[32];
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int w = 0; w < 32; ++w) t += s_part[w];
        out[0] = (T)t;
    }
}

}  // namespace zs

using namespace zs;

extern "C" {

int zs_iw_objective(int dtype, int estimator, void* cost, void* dlogp, void* dlogq, const void* logp,
                    const void* logq, const void* logp_extra, int64_t K, int64_t B, double grad_scale,
                    zs_stream_t stream) {
    ZS_REQUIRE(logp && logq && K >= 1 && B >= 0, ZS_ERR_ARG);
    ZS_REQUIRE(estimator == ZS_EST_SGVB || estimator == ZS_EST_VIMCO || estimator == ZS_EST_ELBO, ZS_ERR_ARG);
    ZS_REQUIRE(!(estimator == ZS_EST_VIMCO && K < 2), ZS_ERR_ARG);
    if (B == 0) return ZS_OK;
    int cols, slices;
    column_geometry(B, cols, slices);
    dim3 block(cols, slices);
    const int64_t grid = (B + cols - 1) / cols;
    ZS_REQUIRE(grid < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);
    cudaStream_t st = as_stream(stream);
    const size_t smem = OBJ_THREADS * (sizeof(double) + sizeof(long long));
    ZS_DTYPE_SWITCH(dtype, {
        auto kern = estimator == ZS_EST_SGVB   ? k_iw_objective<T, ZS_EST_SGVB>
                    : estimator == ZS_EST_ELBO ? k_iw_objective<T, ZS_EST_ELBO>
                                               : k_iw_objective<T, ZS_EST_VIMCO>;
        kern<<<(unsigned)grid, block, smem, st>>>((T*)cost, (T*)dlogp, (T*)dlogq, (const T*)logp, (const T*)logq,
                                                  (const T*)logp_extra, K, B, (T)grad_scale, cols, slices);
    })
    ZS_LAUNCH_CHECK("k_iw_objective");
    return ZS_OK;
}

static int lme_launch(int dtype, bool bwd, void* out, const void* g, const void* x, int64_t K, int64_t B,
                      zs_stream_t stream) {
    ZS_REQUIRE(out && x && K >= 1 && B >= 0, ZS_ERR_ARG);
    if (B == 0) return ZS_OK;
    int cols, slices;
    column_geometry(B, cols, slices);
    dim3 block(cols, slices);
    const int64_t grid = (B + cols - 1) / cols;
    ZS_REQUIRE(grid < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);
    cudaStream_t st = as_stream(stream);
    ZS_DTYPE_SWITCH(dtype, {
        const size_t smem = OBJ_THREADS * sizeof(T);
        if (bwd)
            k_log_mean_exp<T, true><<<(unsigned)grid, block, smem, st>>>((T*)out, (const T*)g, (const T*)x, K, B, cols,
                                                                          slices);
        else
            k_log_mean_exp<T, false><<<(unsigned)grid, block, smem, st>>>((T*)out, nullptr, (const T*)x, K, B, cols,
                                                                           slices);
    })
    ZS_LAUNCH_CHECK("k_log_mean_exp");
    return ZS_OK;
}

int zs_scale_inplace(int dtype, void* buf0, int64_t n0, void* buf1, int64_t n1, void* buf2, int64_t n2,
                     const void* scale_dev, zs_stream_t stream) {
    ZS_REQUIRE(buf0 && scale_dev && n0 >= 0 && n1 >= 0 && n2 >= 0, ZS_ERR_ARG);
    ZS_REQUIRE(aligned16(buf0) && aligned16(buf1) && aligned16(buf2), ZS_ERR_ALIGN);
    int64_t n = n0;
    if (buf1 && n1 > n) n = n1;
    if (buf2 && n2 > n) n = n2;
    if (n == 0) return ZS_OK;
    const int grid = grid_for(n / 4 + 1, 256, 8);
    ZS_DTYPE_SWITCH(dtype, {
        launch_pdl(PDL_SCALE, k_scale_inplace<T>, dim3(grid), dim3(256), 0, as_stream(stream), (T*)buf0, n0, (T*)buf1, n1,
                   (T*)buf2, n2, (const T*)scale_dev);
    })
    ZS_LAUNCH_CHECK("k_scale_inplace");
    return ZS_OK;
}

int zs_combine_sums(int dtype, void* out, const void* a, int64_t na, double scale_a, const void* b, int64_t nb,
                    double scale_b, zs_stream_t stream) {
    ZS_REQUIRE(out && na >= 0 && nb >= 0 && (a || na == 0) && (b || nb == 0), ZS_ERR_ARG);
    ZS_DTYPE_SWITCH(dtype, {
        k_combine_sums<T><<<1, 1024, 0, as_stream(stream)>>>((T*)out, (const T*)a, na, (T)scale_a, (const T*)b, nb,
                                                              (T)scale_b);
    })
    ZS_LAUNCH_CHECK("k_combine_sums");
    return ZS_OK;
}

int zs_log_mean_exp(int dtype, void* out, const void* x, int64_t K, int64_t B, zs_stream_t stream) {
    return lme_launch(dtype, false, out, nullptr, x, K, B, stream);
}

int zs_log_mean_exp_bwd(int dtype, void* dx, const void* g, const void* x, int64_t K, int64_t B,
                        zs_stream_t stream) {
    ZS_REQUIRE(g != nullptr, ZS_ERR_ARG);
    return lme_launch(dtype, true, dx, g, x, K, B, stream);
}

int zs_reinforce_step(int dtype, void* cost, void* dlogp, void* dlogq, float* moving_mean, int* local_step,
                      const void* logp, const void* logq, int64_t N, double decay, double grad_scale,
                      zs_stream_t stream) {
    ZS_REQUIRE(cost && moving_mean && local_step && logp && logq && N >= 1, ZS_ERR_ARG);
    ZS_DTYPE_SWITCH(dtype, {
        k_reinforce<T><<<RF_CLUSTER, RF_THREADS, 0, as_stream(stream)>>>((T*)cost, (T*)dlogp, (T*)dlogq, moving_mean,
                                                                          local_step, (const T*)logp, (const T*)logq, N,
                                                                          (float)decay, (T)grad_scale);
    })
    ZS_LAUNCH_CHECK("k_reinforce");
    return ZS_OK;
}

}  // extern "C"
