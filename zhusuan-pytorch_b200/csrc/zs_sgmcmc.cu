// SG-MCMC parameter updates across parallel chains: one fused pass per update (w_out may alias w) with the
// Gaussian term drawn in-register from Philox (or injected for parity tests).
//
// Replaces (reference file:line):
//   SGLD._update   zhusuan/mcmc/SGLD.py:42-54    w += 0.5*lr*g + N(0, lr)
//   PSGLD._update  zhusuan/mcmc/SGLD.py:67-82    RMSprop-preconditioned SGLD
//   SGHMC._update  zhusuan/mcmc/SGHMC.py:25-56   first / second order, velocity resampling
// The reference draws every noise tensor on the CPU and copies it to the device
// (SGLD.py:51, SGHMC.py:27,33,34) and runs 3-6 elementwise kernels per tensor.
// Scalar coefficients are rounded exactly as the reference's Python does: SGLD.lr is a float32
// 0-d tensor (SGLD.py:20), SGHMC.lr / alpha / beta are Python floats cast to the tensor dtype.
#include "zs_common.cuh"
#include "zs_philox.cuh"

namespace zs {

template <typename T>
struct Quad {
    T v[4];
};

template <typename T>
__device__ __forceinline__ Quad<T> ld4(const T* p);
template <>
__device__ __forceinline__ Quad<float> ld4<float>(const float* p) {
    Pack<float> a = ld_pack(p);
    return Quad<float>{{a.v[0], a.v[1], a.v[2], a.v[3]}};
}
template <>
__device__ __forceinline__ Quad<double> ld4<double>(const double* p) {
    Pack<double> a = ld_pack(p), b = ld_pack(p + 2);
    return Quad<double>{{a.v[0], a.v[1], b.v[0], b.v[1]}};
}
__device__ __forceinline__ void st4(float* p, const Quad<float>& q) {
    Pack<float> a{{q.v[0], q.v[1], q.v[2], q.v[3]}};
    st_pack(p, a);
}
__device__ __forceinline__ void st4(double* p, const Quad<double>& q) {
    Pack<double> a{{q.v[0], q.v[1]}}, b{{q.v[2], q.v[3]}};
    st_pack(p, a);
    st_pack(p + 2, b);
}

// The reference evaluates every update as a chain of separate torch ops (SGLD.py:50-52, SGHMC.py:46-56): each product
// and sum is rounded on its own.  The bodies below spell the roundings out (no fused multiply-add contraction), so the
// single-tensor and the multi-tensor kernels -- different code around the same body -- agree bit for bit.
__device__ __forceinline__ float rmul(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double rmul(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float radd(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double radd(double a, double b) { return __dadd_rn(a, b); }

// Generic driver: Body::apply(i-th element state...) over n elements, 4 per thread.
// VEC requires 16-byte aligned pointers; the last n%4 elements always take the scalar path.
template <typename T, typename Body, bool VEC>
__global__ void __launch_bounds__(256) k_chain_update(Body body, int64_t n, uint64_t seed, uint64_t offset,
                                                      unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const int64_t nq = (n + 3) / 4;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (int64_t)gridDim.x * blockDim.x) {
        float xi[4] = {0.f, 0.f, 0.f, 0.f};
        if (body.needs_rng()) philox_normal4((uint64_t)q, offset, seed, xi);
        const int64_t i0 = q * 4;
        if (VEC && i0 + 4 <= n) {
            body.vec(i0, xi);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (i0 + j < n) body.one(i0 + j, xi[j]);
        }
    }
}

template <typename T>
struct SgldBody {
    T* wo;
    const T* w;
    const T* g;
    const T* noise;  // already scaled, or null
    T half_lr;       // (T)(0.5f * (float)lr)
    float std;       // sqrt(lr)
    __host__ __device__ bool needs_rng() const { return noise == nullptr; }
    __host__ __device__ void bind(const zs_chain_tensor& c) {
        wo = (T*)c.w_out; w = (const T*)c.w; g = (const T*)c.g; noise = (const T*)c.noise;
    }
    bool valid(const zs_chain_tensor& c) const { return c.w_out && c.w && c.g; }
    __device__ __forceinline__ T upd(T wv, T gv, T e) const { return radd(radd(wv, rmul(half_lr, gv)), e); }
    __device__ void one(int64_t i, float xi) const {
        T e = noise ? noise[i] : (T)rmul(std, xi);
        wo[i] = upd(w[i], g[i], e);
    }
    __device__ void vec(int64_t i, const float* xi) const {
        Quad<T> wv = ld4(w + i), gv = ld4(g + i), ev;
        if (noise) ev = ld4(noise + i);
#pragma unroll
        for (int j = 0; j < 4; ++j) wv.v[j] = upd(wv.v[j], gv.v[j], noise ? ev.v[j] : (T)rmul(std, xi[j]));
        st4(wo + i, wv);
    }
};

template <typename T>
struct PsgldBody {
    T* wo;
    const T* w;
    T* aux;
    const T* g;
    const T* unit;  // unit normals or null
    T decay, one_m_decay, eps, lr, half_lr;
    __host__ __device__ bool needs_rng() const { return unit == nullptr; }
    __host__ __device__ void bind(const zs_chain_tensor& c) {
        wo = (T*)c.w_out; w = (const T*)c.w; aux = (T*)c.state; g = (const T*)c.g; unit = (const T*)c.noise;
    }
    bool valid(const zs_chain_tensor& c) const { return c.w_out && c.w && c.g && c.state; }
    __device__ __forceinline__ void upd(T& wv, T& av, T gv, T xi) const {
        av = radd(rmul(decay, av), rmul(one_m_decay, rmul(gv, gv)));
        T G = T(1) / radd(eps, Real<T>::sqrt(av));
        T e = rmul(Real<T>::sqrt(rmul(lr, G)), xi);
        wv = radd(radd(wv, rmul(rmul(half_lr, G), gv)), e);
    }
    __device__ void one(int64_t i, float xi) const {
        T wv = w[i], av = aux[i];
        upd(wv, av, g[i], unit ? unit[i] : (T)xi);
        wo[i] = wv;
        aux[i] = av;
    }
    __device__ void vec(int64_t i, const float* xi) const {
        Quad<T> wv = ld4(w + i), av = ld4(aux + i), gv = ld4(g + i), uv;
        if (unit) uv = ld4(unit + i);
#pragma unroll
        for (int j = 0; j < 4; ++j) upd(wv.v[j], av.v[j], gv.v[j], unit ? uv.v[j] : (T)xi[j]);
        st4(wo + i, wv);
        st4(aux + i, av);
    }
};

template <typename T>
struct SghmcPreBody {
    T* wo;
    const T* w;
    T* v;
    const T* v_noise;  // injected resampled velocity, or null
    float std;         // sqrt(lr)
    int resample, second_order;
    __host__ __device__ bool needs_rng() const { return resample && v_noise == nullptr; }
    __host__ __device__ void bind(const zs_chain_tensor& c) {
        wo = (T*)c.w_out; w = (const T*)c.w; v = (T*)c.state; v_noise = (const T*)c.noise;
    }
    bool valid(const zs_chain_tensor& c) const { return c.w_out && c.w && c.state; }
    __device__ __forceinline__ void upd(T& wv, T& vv, T fresh) const {
        if (resample) vv = fresh;
        if (second_order) wv = radd(wv, rmul(T(0.5), vv));
    }
    __device__ void one(int64_t i, float xi) const {
        T wv = w[i], vv = v[i];
        upd(wv, vv, v_noise ? v_noise[i] : (T)rmul(std, xi));
        if (resample) v[i] = vv;
        if (second_order) wo[i] = wv;
    }
    __device__ void vec(int64_t i, const float* xi) const {
        Quad<T> wv = ld4(w + i), vv = ld4(v + i), nv;
        if (v_noise) nv = ld4(v_noise + i);
#pragma unroll
        for (int j = 0; j < 4; ++j) upd(wv.v[j], vv.v[j], v_noise ? nv.v[j] : (T)rmul(std, xi[j]));
        if (resample) st4(v + i, vv);
        if (second_order) st4(wo + i, wv);
    }
};

template <typename T>
struct SghmcPostBody {
    T* wo;
    const T* w;
    T* v;
    const T* g;
    const T* noise;  // already scaled, or null
    T one_m_alpha, lr, decay_half;
    float std;  // sqrt(2 (alpha-beta) lr)
    int second_order;
    __host__ __device__ bool needs_rng() const { return noise == nullptr; }
    __host__ __device__ void bind(const zs_chain_tensor& c) {
        wo = (T*)c.w_out; w = (const T*)c.w; v = (T*)c.state; g = (const T*)c.g; noise = (const T*)c.noise;
    }
    bool valid(const zs_chain_tensor& c) const { return c.w_out && c.w && c.g && c.state; }
    __device__ __forceinline__ void upd(T& wv, T& vv, T gv, T n) const {
        if (!second_order) {
            vv = radd(radd(rmul(one_m_alpha, vv), rmul(lr, gv)), n);
            wv = radd(wv, vv);
        } else {
            vv = rmul(decay_half, radd(radd(rmul(decay_half, vv), rmul(lr, gv)), n));
            wv = radd(wv, rmul(T(0.5), vv));
        }
    }
    __device__ void one(int64_t i, float xi) const {
        T wv = w[i], vv = v[i];
        upd(wv, vv, g[i], noise ? noise[i] : (T)rmul(std, xi));
        wo[i] = wv;
        v[i] = vv;
    }
    __device__ void vec(int64_t i, const float* xi) const {
        Quad<T> wv = ld4(w + i), vv = ld4(v + i), gv = ld4(g + i), nv;
        if (noise) nv = ld4(noise + i);
#pragma unroll
        for (int j = 0; j < 4; ++j) upd(wv.v[j], vv.v[j], gv.v[j], noise ? nv.v[j] : (T)rmul(std, xi[j]));
        st4(wo + i, wv);
        st4(v + i, vv);
    }
};

template <typename T, typename Body>
static int launch_chain(Body body, int64_t n, bool vec, uint64_t seed, uint64_t offset, void* rng_state,
                        cudaStream_t st, const char* name) {
    if (n == 0) return ZS_OK;
    // injected noise: no draw, the stream position stays
    unsigned long long* rs = body.needs_rng() ? (unsigned long long*)rng_state : nullptr;
    const int grid = grid_for((n + 3) / 4, 256, 64);
    if (vec)
        k_chain_update<T, Body, true><<<grid, 256, 0, st>>>(body, n, seed, offset, rs);
    else
        k_chain_update<T, Body, false><<<grid, 256, 0, st>>>(body, n, seed, offset, rs);
    ZS_LAUNCH_CHECK(name);
    return ZS_OK;
}

// ---- multi-tensor apply: every chain-state tensor of a sampler in ONE launch ---------------------------------
// The table travels in the kernel parameters (graph-capturable, no device allocation).  Tensor t owns the quads
// [qbase[t], qbase[t+1]) of one Philox stream position: element i of tensor t draws word i % 4 of counter
// qbase[t] + i / 4, so a single-tensor call of this entry point equals the single-tensor entry point bit for bit.
constexpr int CHAIN_MAX_TENSORS = ZS_CHAIN_MAX_TENSORS;

struct ChainTable {
    zs_chain_tensor t[CHAIN_MAX_TENSORS];
    long long qbase[CHAIN_MAX_TENSORS + 1];
    unsigned vec_mask;  // bit t: all pointers of tensor t are 16-byte aligned
    int count;
};

template <typename T, typename Body>
__global__ void __launch_bounds__(256) k_chain_update_multi(const __grid_constant__ ChainTable tab, Body proto,
                                                            uint64_t seed, uint64_t offset, unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const long long nq = tab.qbase[tab.count];
    for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < nq; q += (long long)gridDim.x * blockDim.x) {
        int t = 0;
        while (t + 1 < tab.count && q >= tab.qbase[t + 1]) ++t;
        Body body = proto;
        body.bind(tab.t[t]);
        float xi[4] = {0.f, 0.f, 0.f, 0.f};
        if (body.needs_rng()) philox_normal4((uint64_t)q, offset, seed, xi);
        const int64_t n = tab.t[t].n, i0 = (int64_t)(q - tab.qbase[t]) * 4;
        if (((tab.vec_mask >> t) & 1u) && i0 + 4 <= n) {
            body.vec(i0, xi);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (i0 + j < n) body.one(i0 + j, xi[j]);
        }
    }
}

template <typename T, typename Body>
static int launch_chain_multi(Body proto, const zs_chain_tensor* tensors, int n_tensors, uint64_t seed, uint64_t offset,
                              void* rng_state, cudaStream_t st, const char* name) {
    if (n_tensors > CHAIN_MAX_TENSORS) {
        set_last_error_msg("multi-tensor SG-MCMC step: more than ZS_CHAIN_MAX_TENSORS tensors; split the call");
        return ZS_ERR_UNSUPPORTED;
    }
    ChainTable tab;
    tab.count = n_tensors;
    tab.vec_mask = 0;
    tab.qbase[0] = 0;
    bool any_rng = false;
    for (int i = 0; i < n_tensors; ++i) {
        const zs_chain_tensor& ct = tensors[i];
        if (ct.n < 0 || (ct.n > 0 && !proto.valid(ct))) {
            set_last_error_msg("multi-tensor SG-MCMC step: null pointer / negative size in the tensor table");
            return ZS_ERR_ARG;
        }
        tab.t[i] = ct;
        tab.qbase[i + 1] = tab.qbase[i] + (ct.n + 3) / 4;
        if (aligned16(ct.w_out) && aligned16(ct.w) && aligned16(ct.g) && aligned16(ct.state) && aligned16(ct.noise))
            tab.vec_mask |= 1u << i;
        Body b = proto;
        b.bind(ct);
        any_rng = any_rng || (ct.n > 0 && b.needs_rng());
    }
    const long long nq = tab.qbase[n_tensors];
    if (nq == 0) return ZS_OK;
    // injected noise everywhere: no draw, the stream position stays
    unsigned long long* rs = any_rng ? (unsigned long long*)rng_state : nullptr;
    k_chain_update_multi<T, Body><<<grid_for(nq, 256, 64), 256, 0, st>>>(tab, proto, seed, offset, rs);
    ZS_LAUNCH_CHECK(name);
    return ZS_OK;
}

}  // namespace zs

using namespace zs;

extern "C" {

int zs_sgld_step(int dtype, void* w_out, const void* w, const void* g, const void* noise, int64_t n, double lr,
                 uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(w_out && w && g && n >= 0 && lr >= 0, ZS_ERR_ARG);
    const float lr_f = (float)lr;
    const float std = (float)sqrt((double)lr_f);
    const bool vec = aligned16(w_out) && aligned16(w) && aligned16(g) && aligned16(noise);
    ZS_DTYPE_SWITCH(dtype, {
        SgldBody<T> b{(T*)w_out, (const T*)w, (const T*)g, (const T*)noise, (T)(0.5f * lr_f), std};
        return launch_chain<T>(b, n, vec, seed, offset, rng_state, as_stream(stream), "sgld");
    })
}

int zs_psgld_step(int dtype, void* w_out, const void* w, void* aux, const void* g, const void* noise_unit, int64_t n,
                  double lr, double decay, double epsilon, uint64_t seed, uint64_t offset, void* rng_state,
                  zs_stream_t stream) {
    ZS_REQUIRE(w_out && w && aux && g && n >= 0 && lr >= 0, ZS_ERR_ARG);
    const float lr_f = (float)lr;
    const bool vec = aligned16(w_out) && aligned16(w) && aligned16(g) && aligned16(aux) && aligned16(noise_unit);
    ZS_DTYPE_SWITCH(dtype, {
        PsgldBody<T> b{(T*)w_out, (const T*)w, (T*)aux, (const T*)g, (const T*)noise_unit,
                       (T)decay, (T)(1.0 - decay), (T)epsilon, (T)lr_f, (T)(0.5f * lr_f)};
        return launch_chain<T>(b, n, vec, seed, offset, rng_state, as_stream(stream), "psgld");
    })
}

int zs_sghmc_pre(int dtype, void* w_out, const void* w, void* v, const void* v_noise, int64_t n, double lr,
                 int resample, int second_order, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(w_out && w && v && n >= 0 && lr >= 0, ZS_ERR_ARG);
    if (!resample && !second_order) return ZS_OK;
    const float std = (float)sqrt(lr);
    const bool vec = aligned16(w_out) && aligned16(w) && aligned16(v) && aligned16(v_noise);
    ZS_DTYPE_SWITCH(dtype, {
        SghmcPreBody<T> b{(T*)w_out, (const T*)w, (T*)v, (const T*)v_noise, std, resample, second_order};
        return launch_chain<T>(b, n, vec, seed, offset, rng_state, as_stream(stream), "sghmc_pre");
    })
}

int zs_sghmc_post(int dtype, void* w_out, const void* w, void* v, const void* g, const void* noise, int64_t n,
                  double lr, double alpha, double beta, int second_order, uint64_t seed, uint64_t offset,
                  void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(w_out && w && v && g && n >= 0 && lr >= 0, ZS_ERR_ARG);
    ZS_REQUIRE(alpha - beta >= 0, ZS_ERR_ARG);
    const float std = (float)sqrt(2.0 * (alpha - beta) * lr);
    const double dh = exp(-0.5 * alpha);
    const bool vec = aligned16(w_out) && aligned16(w) && aligned16(v) && aligned16(g) && aligned16(noise);
    ZS_DTYPE_SWITCH(dtype, {
        SghmcPostBody<T> b{(T*)w_out, (const T*)w, (T*)v, (const T*)g, (const T*)noise, (T)(1.0 - alpha), (T)lr, (T)dh,
                           std, second_order};
        return launch_chain<T>(b, n, vec, seed, offset, rng_state, as_stream(stream), "sghmc_post");
    })
}

int zs_sgmcmc_multi_step(int dtype, int algorithm, const zs_chain_tensor* tensors, int n_tensors, double lr, double a,
                         double b, int resample, int second_order, uint64_t seed, uint64_t offset, void* rng_state,
                         zs_stream_t stream) {
    ZS_REQUIRE(n_tensors >= 0 && (tensors != nullptr || n_tensors == 0) && lr >= 0, ZS_ERR_ARG);
    if (n_tensors == 0) return ZS_OK;
    cudaStream_t st = as_stream(stream);
    const float lr_f = (float)lr;  // SGLD / PSGLD: lr is a float32 0-d tensor in the reference (SGLD.py:20)
    ZS_DTYPE_SWITCH(dtype, {
        switch (algorithm) {
            case ZS_ALG_SGLD: {
                const float std = (float)sqrt((double)lr_f);
                SgldBody<T> p{nullptr, nullptr, nullptr, nullptr, (T)(0.5f * lr_f), std};
                return launch_chain_multi<T>(p, tensors, n_tensors, seed, offset, rng_state, st, "sgld_multi");
            }
            case ZS_ALG_PSGLD: {  // a = decay, b = epsilon
                PsgldBody<T> p{nullptr, nullptr, nullptr, nullptr, nullptr, (T)a, (T)(1.0 - a), (T)b, (T)lr_f,
                               (T)(0.5f * lr_f)};
                return launch_chain_multi<T>(p, tensors, n_tensors, seed, offset, rng_state, st, "psgld_multi");
            }
            case ZS_ALG_SGHMC_PRE: {
                if (!resample && !second_order) return ZS_OK;
                const float std = (float)sqrt(lr);
                SghmcPreBody<T> p{nullptr, nullptr, nullptr, nullptr, std, resample, second_order};
                return launch_chain_multi<T>(p, tensors, n_tensors, seed, offset, rng_state, st, "sghmc_pre_multi");
            }
            case ZS_ALG_SGHMC_POST: {  // a = alpha (friction), b = beta (variance estimate)
                ZS_REQUIRE(a - b >= 0, ZS_ERR_ARG);
                const float std = (float)sqrt(2.0 * (a - b) * lr);
                const double dh = exp(-0.5 * a);
                SghmcPostBody<T> p{nullptr, nullptr, nullptr, nullptr, nullptr, (T)(1.0 - a), (T)lr, (T)dh, std,
                                   second_order};
                return launch_chain_multi<T>(p, tensors, n_tensors, seed, offset, rng_state, st, "sghmc_post_multi");
            }
            default:
                set_last_error_msg("unknown SG-MCMC algorithm");
                return ZS_ERR_ARG;
        }
    })
}

}  // extern "C"
