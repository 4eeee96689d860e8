// Categorical stochastic node.  The reference has no Categorical (name_mapping,
// zhusuan/framework/bn.py:8-19, stops at Uniform) although north_star names it — parity is
// UNPINNED: the oracle is the closed form log_softmax(logits)[x] (oracle/zs_oracle_impl.h).
// API modelled on zhusuan/distributions/bernoulli.py: value = class index (stored in the
// distribution's float dtype), non-reparameterised, batch_shape = logits.shape[:-1].
//   logits [K|1, M, C] (ZS_FULL or ZS_KBCAST), x [K, M] or [M]
#include "zs_common.cuh"
#include "zs_philox.cuh"

namespace zs {

template <int LPR, typename T>
__device__ __forceinline__ T group_max(T v) {
#pragma unroll
    for (int o = LPR / 2; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o, LPR));
    return v;
}

// log-sum-exp of one row, all LPR lanes get the result
template <int LPR, typename T>
__device__ __forceinline__ T row_lse(const T* row, int64_t C, int lane, T& mx_out) {
    T mx = -INFINITY;
    for (int64_t c = lane; c < C; c += LPR) mx = fmax(mx, row[c]);
    mx = group_max<LPR>(mx);
    T s = T(0);
    for (int64_t c = lane; c < C; c += LPR) s += Real<T>::exp(row[c] - mx);
    s = group_sum<LPR>(s);
    mx_out = mx;
    return mx + Real<T>::log(s);
}

template <typename T, int LPR>
__global__ void __launch_bounds__(256) k_cat_logpmf_fwd(T* __restrict__ out, const T* __restrict__ x, int xm,
                                                        const T* __restrict__ logits, int lm, int64_t K, int64_t M,
                                                        int64_t C) {
    const int lane = threadIdx.x % LPR;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    const int64_t ngrp = (int64_t)gridDim.x * blockDim.x / LPR;
    const int64_t R = K * M;
    for (int64_t base = 0; base < R; base += ngrp) {
        const int64_t r = base + grp;
        const bool valid = r < R;
        const int64_t rr = valid ? r : 0;
        const int64_t m = rr % M;
        const T* row = logits + (lm == ZS_FULL ? rr : m) * C;
        T mx;
        T lse = row_lse<LPR>(row, C, lane, mx);
        if (valid && lane == 0) {
            T xv = xm == ZS_FULL ? x[rr] : (xm == ZS_KBCAST ? x[m] : x[0]);
            int64_t idx = (int64_t)xv;
            out[rr] = (idx >= 0 && idx < C) ? row[idx] - lse : (T)(-INFINITY);
        }
    }
}

// FULL logits: dlogits[r,c] = g[r] * (1[c==x_r] - softmax_c)
template <typename T, int LPR>
__global__ void __launch_bounds__(256) k_cat_logpmf_bwd_full(T* __restrict__ dlogits, const T* __restrict__ g,
                                                             const T* __restrict__ x, int xm,
                                                             const T* __restrict__ logits, int64_t K, int64_t M,
                                                             int64_t C) {
    const int lane = threadIdx.x % LPR;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    const int64_t ngrp = (int64_t)gridDim.x * blockDim.x / LPR;
    const int64_t R = K * M;
    for (int64_t base = 0; base < R; base += ngrp) {
        const int64_t r = base + grp;
        const bool valid = r < R;
        const int64_t rr = valid ? r : 0;
        const int64_t m = rr % M;
        const T* row = logits + rr * C;
        T mx;
        T lse = row_lse<LPR>(row, C, lane, mx);
        if (valid) {
            T xv = xm == ZS_FULL ? x[rr] : (xm == ZS_KBCAST ? x[m] : x[0]);
            const int64_t idx = (int64_t)xv;
            const T gv = g[rr];
            for (int64_t c = lane; c < C; c += LPR) {
                T sm = Real<T>::exp(row[c] - lse);
                dlogits[rr * C + c] = gv * ((c == idx ? T(1) : T(0)) - sm);
            }
        }
    }
}

// KBCAST logits: dlogits[m,c] = sum_k g[k,m] 1[c==x_km] - softmax[m,c] * sum_k g[k,m]
template <typename T, int LPR>
__global__ void __launch_bounds__(256) k_cat_logpmf_bwd_kb(T* __restrict__ dlogits, const T* __restrict__ g,
                                                           const T* __restrict__ x, int xm,
                                                           const T* __restrict__ logits, int64_t K, int64_t M,
                                                           int64_t C) {
    const int lane = threadIdx.x % LPR;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / LPR;
    const int64_t ngrp = (int64_t)gridDim.x * blockDim.x / LPR;
    for (int64_t base = 0; base < M; base += ngrp) {
        const int64_t m0 = base + grp;
        const bool valid = m0 < M;
        const int64_t m = valid ? m0 : 0;
        const T* row = logits + m * C;
        T mx;
        T lse = row_lse<LPR>(row, C, lane, mx);
        if (valid) {
            T gsum = T(0);
            for (int64_t k = 0; k < K; ++k) gsum += g[k * M + m];
            for (int64_t c = lane; c < C; c += LPR) {
                T hit = T(0);
                for (int64_t k = 0; k < K; ++k) {
                    T xv = xm == ZS_FULL ? x[k * M + m] : (xm == ZS_KBCAST ? x[m] : x[0]);
                    if ((int64_t)xv == c) hit += g[k * M + m];
                }
                dlogits[m * C + c] = hit - Real<T>::exp(row[c] - lse) * gsum;
            }
        }
    }
}

// inverse-CDF draw, one thread per (k,m)
template <typename T>
__global__ void __launch_bounds__(256) k_cat_sample(T* __restrict__ out, const T* __restrict__ logits, int lm,
                                                    const T* __restrict__ u_in, int64_t K, int64_t M, int64_t C,
                                                    uint64_t seed, uint64_t offset, unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const int64_t R = K * M;
    for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x) {
        const int64_t m = r % M;
        const T* row = logits + (lm == ZS_FULL ? r : m) * C;
        T u;
        if (u_in) {
            u = u_in[r];
        } else {
            float u4[4];
            philox_uniform4((uint64_t)(r >> 2), offset, seed, u4);
            u = (T)u4[r & 3];
        }
        T mx = -INFINITY;
        for (int64_t c = 0; c < C; ++c) mx = fmax(mx, row[c]);
        T s = T(0);
        for (int64_t c = 0; c < C; ++c) s += Real<T>::exp(row[c] - mx);
        const T target = u * s;
        T cum = T(0);
        int64_t idx = C - 1;
        for (int64_t c = 0; c < C; ++c) {
            cum += Real<T>::exp(row[c] - mx);
            if (cum > target) {
                idx = c;
                break;
            }
        }
        out[r] = (T)idx;
    }
}

}  // namespace zs

using namespace zs;

#define ZS_CAT_SWITCH(dtype, C, ...)                                  \
    ZS_DTYPE_SWITCH(dtype, {                                          \
        if ((C) <= 16) { constexpr int LPR = 4; __VA_ARGS__ }         \
        else { constexpr int LPR = 32; __VA_ARGS__ }                  \
    })

extern "C" {

int zs_categorical_sample(int dtype, void* out, const void* logits, int logits_mode, const void* u_in, int64_t K,
                          int64_t M, int64_t C, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(out && logits && K >= 0 && M >= 0 && C >= 1, ZS_ERR_ARG);
    unsigned long long* rs = u_in ? nullptr : (unsigned long long*)rng_state;  // injected uniforms: no draw
    ZS_REQUIRE(logits_mode == ZS_FULL || logits_mode == ZS_KBCAST, ZS_ERR_ARG);
    if (K * M == 0) return ZS_OK;
    const int grid = grid_for(K * M, 256);
    ZS_DTYPE_SWITCH(dtype, {
        k_cat_sample<T><<<grid, 256, 0, as_stream(stream)>>>((T*)out, (const T*)logits, logits_mode, (const T*)u_in, K,
                                                              M, C, seed, offset, rs);
    })
    ZS_LAUNCH_CHECK("k_cat_sample");
    return ZS_OK;
}

int zs_categorical_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* logits, int logits_mode,
                              int64_t K, int64_t M, int64_t C, zs_stream_t stream) {
    ZS_REQUIRE(out && x && logits && K >= 0 && M >= 0 && C >= 1, ZS_ERR_ARG);
    ZS_REQUIRE(valid_mode(x_mode) && (logits_mode == ZS_FULL || logits_mode == ZS_KBCAST), ZS_ERR_ARG);
    if (K * M == 0) return ZS_OK;
    ZS_CAT_SWITCH(dtype, C, {
        const int grid = grid_for(K * M, 256 / LPR, 256);
        k_cat_logpmf_fwd<T, LPR><<<grid, 256, 0, as_stream(stream)>>>((T*)out, (const T*)x, x_mode, (const T*)logits,
                                                                       logits_mode, K, M, C);
    })
    ZS_LAUNCH_CHECK("k_cat_logpmf_fwd");
    return ZS_OK;
}

int zs_categorical_logpmf_bwd(int dtype, void* dlogits, const void* g, const void* x, int x_mode, const void* logits,
                              int logits_mode, int64_t K, int64_t M, int64_t C, zs_stream_t stream) {
    ZS_REQUIRE(dlogits && g && x && logits && K >= 0 && M >= 0 && C >= 1, ZS_ERR_ARG);
    ZS_REQUIRE(valid_mode(x_mode) && (logits_mode == ZS_FULL || logits_mode == ZS_KBCAST), ZS_ERR_ARG);
    if (K * M == 0) return ZS_OK;
    ZS_CAT_SWITCH(dtype, C, {
        if (logits_mode == ZS_FULL) {
            const int grid = grid_for(K * M, 256 / LPR, 256);
            k_cat_logpmf_bwd_full<T, LPR><<<grid, 256, 0, as_stream(stream)>>>((T*)dlogits, (const T*)g, (const T*)x,
                                                                                x_mode, (const T*)logits, K, M, C);
        } else {
            const int grid = grid_for(M, 256 / LPR, 256);
            k_cat_logpmf_bwd_kb<T, LPR><<<grid, 256, 0, as_stream(stream)>>>((T*)dlogits, (const T*)g, (const T*)x,
                                                                              x_mode, (const T*)logits, K, M, C);
        }
    })
    ZS_LAUNCH_CHECK("k_cat_logpmf_bwd");
    return ZS_OK;
}

}  // extern "C"
