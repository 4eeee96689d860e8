// Fused latent-node kernels: everything a latent stochastic node contributes to one objective step,
// in one launch forward and one launch backward.
//
// forward  : z ~ q (Philox in-kernel or injected noise), log q(z) and log p(z) under the prior,
//            both summed over the event axis E.
//            Replaces Normal._sample (normal.py:89-107) + Normal._log_prob twice (normal.py:109-126,
//            once in the variational net, once for the generator's prior, iwae.py:60-72,102-120) + the
//            event sums (base.py:175-176, stochastic_tensor.py:164-165); for Bernoulli latents
//            Bernoulli._sample / _log_prob (bernoulli.py:72-95).
// backward : gradient of (dlogq . log q + dlogp . log p + <dz_up, z>) wrt the variational parameters:
//            the autograd backward of both log-densities, the upstream gradient of the sample coming
//            back from the decoder, and the pathwise backward of the sample through `.repeat`
//            (a sum over the K particles), fused.
// Both are specialised for what the hot path uses: float4-aligned event rows (E % 4 == 0), variational
// parameters FULL or KBCAST, prior parameters KBCAST (or NULL = the standard prior) without gradient.
// Anything else returns ZS_ERR_UNSUPPORTED and the caller composes the general kernels of zs_nodes.cu.
#include <initializer_list>
#include <stdlib.h>
#include <type_traits>

#include "zs_common.cuh"
#include "zs_philox.cuh"

namespace zs {

template <typename T>
struct V4 {
    T v[4];
};

template <typename T>
__device__ __forceinline__ V4<T> ldv4(const T* p);
template <>
__device__ __forceinline__ V4<float> ldv4<float>(const float* p) {
    const float4 a = *reinterpret_cast<const float4*>(p);
    return V4<float>{{a.x, a.y, a.z, a.w}};
}
template <>
__device__ __forceinline__ V4<double> ldv4<double>(const double* p) {
    const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2);
    return V4<double>{{a.x, a.y, b.x, b.y}};
}
__device__ __forceinline__ void stv4(float* p, const V4<float>& q) {
    *reinterpret_cast<float4*>(p) = make_float4(q.v[0], q.v[1], q.v[2], q.v[3]);
}
__device__ __forceinline__ void stv4(double* p, const V4<double>& q) {
    *reinterpret_cast<double2*>(p) = make_double2(q.v[0], q.v[1]);
    *reinterpret_cast<double2*>(p + 2) = make_double2(q.v[2], q.v[3]);
}

constexpr int FAM_NORMAL = 0, FAM_BERNOULLI = 1;

template <typename T>
__device__ __forceinline__ T normal_c() {
    return (T)(-0.9189385332046727);
}

// Parameter-only transcendentals.  They are redone by every k-slice of a row, so for float they go to the SFU:
// lg2.approx has an absolute error of 2^-22 in log2 units on [0.5, 2] and <= 2 ulp elsewhere, rcp.approx <= 1 ulp --
// both far inside the 1e-5 parity budget of a 40-term row sum.  double keeps libm / IEEE division.
__device__ __forceinline__ float lat_log(float x) { return fast_log2(x) * 0.6931471805599453f; }
__device__ __forceinline__ double lat_log(double x) { return ::log(x); }
__device__ __forceinline__ float lat_rcp(float x) { return fast_rcp(x); }
__device__ __forceinline__ double lat_rcp(double x) { return 1.0 / x; }

// ---------------------------------------------------------------------------------------------
// forward: G lanes per batch row m; lane j owns float4 units j, j+G, ... of the row.  For KBCAST
// parameters the group keeps mean / std / log std / precision of its units in registers and walks
// the particles k = ks, ks+KS, ... — the transcendental work on the parameters is done once per
// (m, e), not once per particle.  UPL = units per lane held in registers (E/4 <= G*UPL).
// ---------------------------------------------------------------------------------------------
template <typename T>
struct UnitParams {
    V4<T> a, b, logb, prec;        // variational: mean, std, log std, exp(-2 log std)  (Bernoulli: a = probs)
    V4<T> pa, plogb, pprec;        // prior: mean, log std, precision                 (Bernoulli: pa = probs)
};

template <typename T, int FAM>
__device__ __forceinline__ void load_unit_params(UnitParams<T>& u, const T* a, const T* b, const T* pa, const T* pb,
                                                 int64_t idx, int64_t kidx) {
    u.a = ldv4(a + idx);
    if (FAM == FAM_NORMAL) {
        u.b = ldv4(b + idx);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            u.logb.v[q] = lat_log(u.b.v[q]);
            // exp(-2 log std) of normal.py:122 is 1 / std^2 to within an ulp
            u.prec.v[q] = lat_rcp(u.b.v[q] * u.b.v[q]);
        }
        if (pa) u.pa = ldv4(pa + kidx);
        else u.pa = V4<T>{{T(0), T(0), T(0), T(0)}};
        if (pb) {
            const V4<T> ps = ldv4(pb + kidx);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                u.plogb.v[q] = lat_log(ps.v[q]);
                u.pprec.v[q] = lat_rcp(ps.v[q] * ps.v[q]);
            }
        } else {
            // standard prior: log(1) = 0 and exp(-2*0) = 1 exactly, as the reference computes them
            u.plogb = V4<T>{{T(0), T(0), T(0), T(0)}};
            u.pprec = V4<T>{{T(1), T(1), T(1), T(1)}};
        }
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {  // log(p + 1e-8), log((1-p) + 1e-8) of bernoulli.py:94
            u.logb.v[q] = lat_log(u.a.v[q] + T(1e-8));
            u.prec.v[q] = lat_log((T(1) - u.a.v[q]) + T(1e-8));
        }
        if (pa) u.pa = ldv4(pa + kidx);
        else u.pa = V4<T>{{T(0.5), T(0.5), T(0.5), T(0.5)}};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            u.plogb.v[q] = lat_log(u.pa.v[q] + T(1e-8));
            u.pprec.v[q] = lat_log((T(1) - u.pa.v[q]) + T(1e-8));
        }
    }
}

template <typename T, int FAM, int G>
__global__ void __launch_bounds__(256)
    k_latent_fwd(T* __restrict__ z, T* __restrict__ logq, T* __restrict__ logp, const T* __restrict__ a,
                 int a_mode, const T* __restrict__ b, int b_mode, const T* __restrict__ pa, const T* __restrict__ pb,
                 const T* __restrict__ noise_in, int64_t K, int64_t M, int64_t E, int KS, uint64_t seed,
                 uint64_t offset, unsigned long long* rs) {
    offset = rng_acquire(offset, rs, nullptr, true);
    const int lane = threadIdx.x % G;
    const int64_t grp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) / G;  // group -> (m, k-slice)
    const int64_t E4 = E >> 2;
    const int64_t m = grp / KS;
    const int ks = (int)(grp % KS);
    const bool valid = m < M;
    const bool kb = a_mode == ZS_KBCAST;
    // all lanes of a group run the same trip counts (the group shuffles below need every lane)
    for (int64_t j0 = 0; j0 < E4; j0 += G) {
        const int64_t j = j0 + lane;
        const bool active = valid && j < E4;
        UnitParams<T> up;
        if (active && kb) load_unit_params<T, FAM>(up, a, b, pa, pb, m * E + 4 * j, m * E + 4 * j);
        const int64_t trips = (K + KS - 1) / KS;  // uniform across the warp: the shuffles need every lane
        for (int64_t t = 0; t < trips; ++t) {
            const int64_t k = ks + t * KS;
            T accq = T(0), accp = T(0);
            if (active && k < K) {
                const int64_t r = k * M + m, fe = r * E + 4 * j;
                if (!kb) load_unit_params<T, FAM>(up, a, b, pa, pb, fe, m * E + 4 * j);
                V4<T> nz;
                if (noise_in) {
                    nz = ldv4(noise_in + fe);
                } else {
                    float n4[4];  // one Philox counter per float4 unit (element i: counter i/4, word i%4)
                    if (FAM == FAM_NORMAL) philox_normal4((uint64_t)(fe >> 2), offset, seed, n4);
                    else philox_uniform4((uint64_t)(fe >> 2), offset, seed, n4);
#pragma unroll
                    for (int q = 0; q < 4; ++q) nz.v[q] = (T)n4[q];
                }
                V4<T> zv;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (FAM == FAM_NORMAL) {
                        const T zz = up.a.v[q] + up.b.v[q] * nz.v[q];  // normal.py:105
                        zv.v[q] = zz;
                        const T d = zz - up.a.v[q];                     // normal.py:121-124 at the sample
                        accq += (normal_c<T>() - up.logb.v[q]) - (T(0.5) * up.prec.v[q]) * (d * d);
                        const T dp = zz - up.pa.v[q];
                        accp += (normal_c<T>() - up.plogb.v[q]) - (T(0.5) * up.pprec.v[q]) * (dp * dp);
                    } else {
                        const T zz = nz.v[q] < up.a.v[q] ? T(1) : T(0);  // bernoulli.py:79
                        zv.v[q] = zz;
                        accq += zz * up.logb.v[q] + (T(1) - zz) * up.prec.v[q];    // bernoulli.py:94
                        accp += zz * up.plogb.v[q] + (T(1) - zz) * up.pprec.v[q];
                    }
                }
                stv4(z + fe, zv);
            }
            // E4 <= G is the common case (one pass): the row sum is complete after the group reduction;
            // longer rows accumulate across passes through the output (zeroed by the first pass)
            accq = group_sum<G>(accq);
            accp = group_sum<G>(accp);
            if (valid && lane == 0 && k < K) {
                const int64_t r = k * M + m;
                if (logq) logq[r] = (j0 == 0 ? T(0) : logq[r]) + accq;
                if (logp) logp[r] = (j0 == 0 ? T(0) : logp[r]) + accp;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// forward, packed rows (E/4 <= 32, the hot-path case: Z = 40 -> 10 units).  ncu on the kernel above at config 2:
// 11.0 M warp instructions with 22 of 32 lanes active (10 of the 16 lanes of a group own a unit) and the
// parameter transcendentals redone by 16 k-slices per row -- issue-bound at 17.5 us for 8 MB of output.  Here a warp
// packs RW = 32 / (E/4) rows (30 of 32 lanes busy at Z = 40), row sums are segmented shuffle reductions
// (no shared memory, fixed order), a thread keeps its unit's parameters for all its particles
// k = ks, ks + KS, ... (gridDim.y = KS slices with equal trip counts) and works on two particles at a time so two
// Philox / Box-Muller chains are in flight.
// ---------------------------------------------------------------------------------------------
template <typename T, int FAM>
__device__ __forceinline__ void latent_unit(const UnitParams<T>& up, const T* __restrict__ noise_in, T* __restrict__ z,
                                            int64_t fe, uint64_t seed, uint64_t offset, T& accq, T& accp) {
    V4<T> nz;
    if (noise_in) {
        nz = ldv4(noise_in + fe);
    } else {
        float n4[4];  // one Philox counter per float4 unit (element i: counter i/4, word i%4)
        if (FAM == FAM_NORMAL) philox_normal4((uint64_t)(fe >> 2), offset, seed, n4);
        else philox_uniform4((uint64_t)(fe >> 2), offset, seed, n4);
#pragma unroll
        for (int q = 0; q < 4; ++q) nz.v[q] = (T)n4[q];
    }
    V4<T> zv;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        if (FAM == FAM_NORMAL) {
            const T zz = up.a.v[q] + up.b.v[q] * nz.v[q];  // normal.py:105
            zv.v[q] = zz;
            const T d = zz - up.a.v[q];                     // normal.py:121-124 at the sample
            accq += (normal_c<T>() - up.logb.v[q]) - (T(0.5) * up.prec.v[q]) * (d * d);
            const T dp = zz - up.pa.v[q];
            accp += (normal_c<T>() - up.plogb.v[q]) - (T(0.5) * up.pprec.v[q]) * (dp * dp);
        } else {
            const T zz = nz.v[q] < up.a.v[q] ? T(1) : T(0);  // bernoulli.py:79
            zv.v[q] = zz;
            accq += zz * up.logb.v[q] + (T(1) - zz) * up.prec.v[q];    // bernoulli.py:94
            accp += zz * up.plogb.v[q] + (T(1) - zz) * up.pprec.v[q];
        }
    }
    stv4(z + fe, zv);
}

// sum over the E4 consecutive lanes of a row; valid in the row's first lane (j == 0)
template <typename T>
__device__ __forceinline__ T segment_sum(T v, int j, int E4) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const T other = __shfl_down_sync(0xffffffffu, v, o);
        if (j + o < E4) v += other;
    }
    return v;
}

constexpr int LF_WARPS = 4;

template <typename T, int FAM>
__global__ void __launch_bounds__(LF_WARPS * 32)
    k_latent_fwd_packed(T* __restrict__ z, T* __restrict__ logq, T* __restrict__ logp, const T* __restrict__ a,
                        int a_mode, const T* __restrict__ b, const T* __restrict__ pa, const T* __restrict__ pb,
                        const T* __restrict__ noise_in, int K, int64_t M, int E4, int RW, int KS, uint64_t seed,
                        uint64_t offset, unsigned long long* rs) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rl = lane / E4, j = lane - rl * E4;
    const int64_t m = ((int64_t)blockIdx.x * LF_WARPS + warp) * RW + rl;
    const bool active = rl < RW && m < M;
    const int64_t E = 4 * (int64_t)E4, ME = M * E;
    const bool kb = a_mode == ZS_KBCAST;
    const int64_t pidx = m * E + 4 * j;  // the unit inside [M,E]
    UnitParams<T> up;
    if (active && kb) load_unit_params<T, FAM>(up, a, b, pa, pb, pidx, pidx);
    // the stream position is read by the CTA's leader while the other warps load and prepare their parameters
    offset = rng_acquire(offset, rs, nullptr, true);
    // every slice runs the same trip count (the shuffles need the whole warp); particles past K are skipped
    const int trips = (K + KS - 1) / KS;
    for (int t = 0; t < trips; t += 2) {
        const int k0 = (int)blockIdx.y + t * KS, k1 = k0 + KS;
        const bool on0 = active && k0 < K, on1 = active && t + 1 < trips && k1 < K;
        T q0 = T(0), p0 = T(0), q1 = T(0), p1 = T(0);
        if (on0) {
            const int64_t fe = (int64_t)k0 * ME + pidx;
            if (!kb) load_unit_params<T, FAM>(up, a, b, pa, pb, fe, pidx);
            latent_unit<T, FAM>(up, noise_in, z, fe, seed, offset, q0, p0);
        }
        if (on1) {
            const int64_t fe = (int64_t)k1 * ME + pidx;
            if (!kb) load_unit_params<T, FAM>(up, a, b, pa, pb, fe, pidx);
            latent_unit<T, FAM>(up, noise_in, z, fe, seed, offset, q1, p1);
        }
        q0 = segment_sum(q0, j, E4);
        p0 = segment_sum(p0, j, E4);
        q1 = segment_sum(q1, j, E4);
        p1 = segment_sum(p1, j, E4);
        if (j == 0) {
            if (on0) {
                if (logq) logq[(int64_t)k0 * M + m] = q0;
                if (logp) logp[(int64_t)k0 * M + m] = p0;
            }
            if (on1) {
                if (logq) logq[(int64_t)k1 * M + m] = q1;
                if (logp) logp[(int64_t)k1 * M + m] = p1;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// forward, the hot configuration (float, KBCAST parameters, E/4 <= 32, everything indexable in 32 bits): the packed
// kernel above executed ~350 instructions per float4 of latents (ncu round 2: 6.3 M warp instructions for 512 k
// float4, issue-bound at 11 us).  This one is written for instruction count:
//   * every parameter-only term is reduced to what the particle loop needs: the per-row constant
//     sum_q (c - log std_q) is added once, the loop keeps 0.5/std_q^2 (Normal) or the two logs (Bernoulli);
//   * a standard prior (STDP) contributes E*c - 0.5 sum z^2 (Normal) or E*log(0.5 + 1e-8) (Bernoulli(0.5):
//     both branches of bernoulli.py:94 are the same number) -- no prior registers, one FMA per element;
//   * 32-bit index arithmetic, lane -> (row, unit) by a multiply-shift instead of an integer division,
//     the segmented row sums skip the shuffle levels wider than a row;
//   * Box-Muller on the SFU (zs_philox.cuh).
// Sums are re-associated against the reference's elementwise order (a float32 rounding-level difference, 1e-7
// relative; the parity budget is 1e-5).
// ---------------------------------------------------------------------------------------------
template <int FAM, bool STDP>
__global__ void __launch_bounds__(LF_WARPS * 32, 8)
    k_latent_fwd_fast(float* __restrict__ z, float* __restrict__ logq, float* __restrict__ logp,
                      const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ pa,
                      const float* __restrict__ pb, const float* __restrict__ noise_in, int K, int M, int E4, int RW,
                      int KS, unsigned inv_e4, uint64_t seed, uint64_t offset, unsigned long long* rs,
                      unsigned char* __restrict__ zbits) {
    pdl_wait();     // the parameters may come from the kernel before this one
    pdl_trigger();  // the next kernel's CTAs may be scheduled as this grid drains
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int rl = (int)(((unsigned)lane * inv_e4) >> 16), j = lane - rl * E4;  // lane / E4, lane % E4
    const int m = ((int)blockIdx.x * LF_WARPS + warp) * RW + rl;
    const bool active = rl < RW && m < M;
    const int E = 4 * E4;
    const unsigned ME4 = (unsigned)M * (unsigned)E4;   // float4 units per particle
    const unsigned punit = (unsigned)m * (unsigned)E4 + (unsigned)j;  // this thread's unit inside [M, E/4]
    // ---- per-unit constants
    float4 av = make_float4(0.f, 0.f, 0.f, 0.f), bv = av, h = av, l0 = av, l1 = av;
    float cq = 0.f, cp = 0.f;  // particle-independent parts of this unit's log q / log p
    float4 pm = av, hp = av;
    if (active) {
        av = *reinterpret_cast<const float4*>(a + 4 * (size_t)punit);
        if (FAM == FAM_NORMAL) {
            bv = *reinterpret_cast<const float4*>(b + 4 * (size_t)punit);
            const float c = normal_c<float>();
            cq = (c - lat_log(bv.x)) + (c - lat_log(bv.y)) + (c - lat_log(bv.z)) + (c - lat_log(bv.w));
            h = make_float4(0.5f * lat_rcp(bv.x * bv.x), 0.5f * lat_rcp(bv.y * bv.y), 0.5f * lat_rcp(bv.z * bv.z),
                            0.5f * lat_rcp(bv.w * bv.w));
            if (STDP) {
                cp = 4.0f * c;
            } else {
                if (pa) pm = *reinterpret_cast<const float4*>(pa + 4 * (size_t)punit);
                float4 ps = make_float4(1.f, 1.f, 1.f, 1.f);
                if (pb) ps = *reinterpret_cast<const float4*>(pb + 4 * (size_t)punit);
                cp = (c - lat_log(ps.x)) + (c - lat_log(ps.y)) + (c - lat_log(ps.z)) + (c - lat_log(ps.w));
                hp = make_float4(0.5f * lat_rcp(ps.x * ps.x), 0.5f * lat_rcp(ps.y * ps.y), 0.5f * lat_rcp(ps.z * ps.z),
                                 0.5f * lat_rcp(ps.w * ps.w));
            }
        } else {
            // log(p + 1e-8), log((1-p) + 1e-8) of bernoulli.py:94: l1 + z (l0 - l1) per element
            l0 = make_float4(lat_log(av.x + 1e-8f), lat_log(av.y + 1e-8f), lat_log(av.z + 1e-8f), lat_log(av.w + 1e-8f));
            l1 = make_float4(lat_log((1.f - av.x) + 1e-8f), lat_log((1.f - av.y) + 1e-8f), lat_log((1.f - av.z) + 1e-8f),
                             lat_log((1.f - av.w) + 1e-8f));
            cq = (l1.x + l1.y) + (l1.z + l1.w);
            l0 = make_float4(l0.x - l1.x, l0.y - l1.y, l0.z - l1.z, l0.w - l1.w);
            if (STDP) {
                cp = 4.0f * lat_log(0.5f + 1e-8f);
            } else {
                const float4 pp = *reinterpret_cast<const float4*>(pa + 4 * (size_t)punit);
                pm = make_float4(lat_log(pp.x + 1e-8f), lat_log(pp.y + 1e-8f), lat_log(pp.z + 1e-8f), lat_log(pp.w + 1e-8f));
                hp = make_float4(lat_log((1.f - pp.x) + 1e-8f), lat_log((1.f - pp.y) + 1e-8f), lat_log((1.f - pp.z) + 1e-8f),
                                 lat_log((1.f - pp.w) + 1e-8f));
                cp = (hp.x + hp.y) + (hp.z + hp.w);
                pm = make_float4(pm.x - hp.x, pm.y - hp.y, pm.z - hp.z, pm.w - hp.w);
            }
        }
    }
    // the stream position is read by the CTA's leader while the other warps prepare their constants
    offset = rng_acquire(offset, rs, nullptr, true);

    auto one = [&](int k, float& accq, float& accp) {
        const unsigned unit = (unsigned)k * ME4 + punit;  // global float4 index == Philox counter of these 4 elements
        float n4[4];
        if (noise_in) {
            const float4 t = *reinterpret_cast<const float4*>(noise_in + 4 * (size_t)unit);
            n4[0] = t.x; n4[1] = t.y; n4[2] = t.z; n4[3] = t.w;
        } else if (FAM == FAM_NORMAL) {
            philox_normal4((uint64_t)unit, offset, seed, n4);
        } else {
            philox_uniform4((uint64_t)unit, offset, seed, n4);
        }
        float4 zv;
        if (FAM == FAM_NORMAL) {
            zv = make_float4(fmaf(bv.x, n4[0], av.x), fmaf(bv.y, n4[1], av.y), fmaf(bv.z, n4[2], av.z),
                             fmaf(bv.w, n4[3], av.w));  // normal.py:105
            const float d0 = zv.x - av.x, d1 = zv.y - av.y, d2 = zv.z - av.z, d3 = zv.w - av.w;  // normal.py:121-124
            accq = cq - ((h.x * (d0 * d0) + h.y * (d1 * d1)) + (h.z * (d2 * d2) + h.w * (d3 * d3)));
            if (STDP) {
                accp = cp - 0.5f * ((zv.x * zv.x + zv.y * zv.y) + (zv.z * zv.z + zv.w * zv.w));
            } else {
                const float e0 = zv.x - pm.x, e1 = zv.y - pm.y, e2 = zv.z - pm.z, e3 = zv.w - pm.w;
                accp = cp - ((hp.x * (e0 * e0) + hp.y * (e1 * e1)) + (hp.z * (e2 * e2) + hp.w * (e3 * e3)));
            }
        } else {
            zv = make_float4(n4[0] < av.x ? 1.f : 0.f, n4[1] < av.y ? 1.f : 0.f, n4[2] < av.z ? 1.f : 0.f,
                             n4[3] < av.w ? 1.f : 0.f);  // bernoulli.py:79
            accq = cq + ((zv.x * l0.x + zv.y * l0.y) + (zv.z * l0.z + zv.w * l0.w));
            if (STDP) accp = cp;
            else accp = cp + ((zv.x * pm.x + zv.y * pm.y) + (zv.z * pm.z + zv.w * pm.w));
        }
        *reinterpret_cast<float4*>(z + 4 * (size_t)unit) = zv;
        // Bernoulli samples are 0 / 1: four of them as one byte per float4 unit, for consumers that only need the
        // pattern (zs_iw_bernoulli_fused_vimco_latent reads 0.5 MB of these instead of 8 MB of floats at config 3)
        if (FAM == FAM_BERNOULLI && zbits)
            zbits[unit] = (unsigned char)((zv.x != 0.f ? 1 : 0) | (zv.y != 0.f ? 2 : 0) | (zv.z != 0.f ? 4 : 0) |
                                          (zv.w != 0.f ? 8 : 0));
    };
    // sum over the E4 consecutive lanes of a row (valid in the row's first lane); levels wider than a row are skipped
    auto row_sum = [&](float v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            if (o < E4) {  // uniform
                const float other = __shfl_down_sync(0xffffffffu, v, o);
                if (j + o < E4) v += other;
            }
        }
        return v;
    };
    const int trips = (K + KS - 1) / KS;  // equal for every slice (the shuffles need the whole warp)
    for (int t = 0; t < trips; t += 2) {
        const int k0 = (int)blockIdx.y + t * KS, k1 = k0 + KS;
        const bool on0 = active && k0 < K, on1 = active && t + 1 < trips && k1 < K;
        float q0 = 0.f, p0 = 0.f, q1 = 0.f, p1 = 0.f;
        if (on0) one(k0, q0, p0);
        if (on1) one(k1, q1, p1);
        q0 = row_sum(q0);
        q1 = row_sum(q1);
        if (logp != nullptr && !(STDP && FAM == FAM_BERNOULLI)) {
            p0 = row_sum(p0);
            p1 = row_sum(p1);
        } else {
            p0 *= (float)E4;  // a constant per unit: E4 units of it
            p1 *= (float)E4;
        }
        if (j == 0) {
            if (on0) {
                if (logq) logq[(unsigned)k0 * (unsigned)M + (unsigned)m] = q0;
                if (logp) logp[(unsigned)k0 * (unsigned)M + (unsigned)m] = p0;
            }
            if (on1) {
                if (logq) logq[(unsigned)k1 * (unsigned)M + (unsigned)m] = q1;
                if (logp) logp[(unsigned)k1 * (unsigned)M + (unsigned)m] = p1;
            }
        }
    }
    (void)E;
}

// ---------------------------------------------------------------------------------------------
// backward: block = LB_X float4 units of [M,E] x blockDim.y particle slices, fixed-order sum over slices.
// Parameter-only terms (precision, 1/std) are hoisted out of the particle loop and take the SFU reciprocal.
// The kernel moves 17 MB at config 2 and was latency-bound (ncu round 1: long_scoreboard 4.35, 1.44 waves of
// 16 x 16 blocks whose threads walked 3-4 particles two at a time): now blockDim.y = ceil(K/2) slices (25 at K = 50),
// every thread owns two particles whose six loads are all issued before the first use, LB_X = 8 units (one 128-byte
// line per particle row) so that 1280 CTAs spread evenly over the SMs.
// ---------------------------------------------------------------------------------------------
constexpr int LB_X_MAX = 8, LB_Y_MAX = 32;

// STDP: the prior is the family's standard one (prior_mean / prior_std NULL): its terms are constants, not registers.
template <typename T, int FAM, bool STDP>
__global__ void __launch_bounds__(LB_X_MAX* LB_Y_MAX, sizeof(T) == 4 ? 4 : 1)
    k_latent_bwd(T* __restrict__ da, T* __restrict__ db, const T* __restrict__ gq, const T* __restrict__ gp,
                 const T* __restrict__ dz_up, const T* __restrict__ z, const T* __restrict__ a, int a_mode,
                 const T* __restrict__ b, int b_mode, const T* __restrict__ pa, const T* __restrict__ pb,
                 int reparam, int64_t K, int64_t M, int64_t E) {
    const int64_t ME4 = (M * E) >> 2;
    const int LBX = blockDim.x, LBY = blockDim.y;
    const int64_t u = (int64_t)blockIdx.x * LBX + threadIdx.x;
    const bool valid = u < ME4;
    const bool full = a_mode == ZS_FULL;  // FULL parameters: per-particle gradients, no reduction
    V4<T> sa{{T(0), T(0), T(0), T(0)}}, sb{{T(0), T(0), T(0), T(0)}};
    if (valid) {
        const int64_t ke = 4 * u, m = ke / E;
        // per unit: a (mean | probs), 1/std (Normal) or the two reciprocals of bernoulli.py:94's autograd; the
        // prior's mean and precision unless STDP.  No logarithms on the backward path.
        V4<T> pa_, r0, r1, pm, pprec;
        auto load_params = [&](int64_t idx) {
            pa_ = ldv4(a + idx);
            if (FAM == FAM_BERNOULLI) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    r0.v[q] = lat_rcp(pa_.v[q] + T(1e-8));
                    r1.v[q] = lat_rcp((T(1) - pa_.v[q]) + T(1e-8));
                }
            } else {
                const V4<T> sd = ldv4(b + idx);
#pragma unroll
                for (int q = 0; q < 4; ++q) r0.v[q] = lat_rcp(sd.v[q]);  // 1/std; exp(-2 log std) = (1/std)^2
                if (!STDP) {
                    if (pa) pm = ldv4(pa + ke);
                    else pm = V4<T>{{T(0), T(0), T(0), T(0)}};
                    if (pb) {
                        const V4<T> ps = ldv4(pb + ke);
#pragma unroll
                        for (int q = 0; q < 4; ++q) pprec.v[q] = lat_rcp(ps.v[q] * ps.v[q]);
                    } else {
                        pprec = V4<T>{{T(1), T(1), T(1), T(1)}};
                    }
                }
            }
        };
        constexpr int LBU = 2;  // particles in flight per thread
        for (int64_t k0 = threadIdx.y; k0 < K; k0 += (int64_t)LBU * LBY) {
            T g_q[LBU], g_p[LBU];
            V4<T> zv[LBU], du[LBU];
#pragma unroll
            for (int i = 0; i < LBU; ++i) {
                const int64_t k = k0 + (int64_t)i * LBY;
                const int64_t kc = k < K ? k : k0;  // always in bounds
                const int64_t r = kc * M + m, fe = kc * (M * E) + ke;
                g_q[i] = gq ? gq[r] : T(0);
                g_p[i] = gp ? gp[r] : T(0);
                zv[i] = ldv4(z + fe);
                if (dz_up && reparam) du[i] = ldv4(dz_up + fe);
                else du[i] = V4<T>{{T(0), T(0), T(0), T(0)}};
            }
            if (!full) load_params(ke);  // loop-invariant: issued after the particle loads, hoisted by the compiler
#pragma unroll
            for (int i = 0; i < LBU; ++i) {
                const int64_t k = k0 + (int64_t)i * LBY;
                if (k >= K) break;
                const int64_t fe = k * (M * E) + ke;
                if (full) load_params(fe);
                V4<T> oa, ob;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    if (FAM == FAM_NORMAL) {
                        // autograd of normal.py:121-124 (same association as NormalOp::grad in zs_nodes.cu)
                        const T rstd = r0.v[q], prec = rstd * rstd, zz = zv[i].v[q];
                        const T d = zz - pa_.v[q];
                        const T dzq = -(g_q[i] * (T(0.5) * prec)) * (T(2) * d);
                        const T dprec = -(g_q[i] * (d * d)) * T(0.5);
                        const T dlogstd = -g_q[i] + (dprec * prec) * T(-2);
                        T dmean = -dzq, dstd = dlogstd * rstd;
                        if (reparam) {
                            T dzp = T(0);
                            if (gp) {
                                if (STDP) dzp = -(g_p[i] * T(0.5)) * (T(2) * zz);
                                else dzp = -(g_p[i] * (T(0.5) * pprec.v[q])) * (T(2) * (zz - pm.v[q]));
                            }
                            const T dzt = (du[i].v[q] + dzp) + dzq;  // total gradient reaching the sample
                            dmean += dzt;                            // z = mean + std*eps
                            dstd += dzt * (d * rstd);                // eps recovered from the sample
                        }
                        oa.v[q] = dmean;
                        ob.v[q] = dstd;
                    } else {
                        // autograd of bernoulli.py:94 wrt probs (samples carry no gradient)
                        const T zz = zv[i].v[q];
                        oa.v[q] = (g_q[i] * zz) * r0.v[q] - (g_q[i] * (T(1) - zz)) * r1.v[q];
                        ob.v[q] = T(0);
                    }
                }
                if (full) {
                    if (da) stv4(da + fe, oa);
                    if (db && FAM == FAM_NORMAL) stv4(db + fe, ob);
                } else {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        sa.v[q] += oa.v[q];
                        sb.v[q] += ob.v[q];
                    }
                }
            }
        }
    }
    if (full) return;
    __shared__ T red[2][LB_Y_MAX][LB_X_MAX][4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        red[0][threadIdx.y][threadIdx.x][q] = sa.v[q];
        red[1][threadIdx.y][threadIdx.x][q] = sb.v[q];
    }
    __syncthreads();
    // fixed-order sum over the slices: thread (x, y < 8) adds up component (y & 3) of array (y >> 2)
    if (threadIdx.y < 8 && valid) {
        const int arr = threadIdx.y >> 2, q = threadIdx.y & 3;
        T t = T(0);
        for (int sl = 0; sl < LBY; ++sl) t += red[arr][sl][threadIdx.x][q];
        T* dst = arr == 0 ? da : (FAM == FAM_NORMAL ? db : nullptr);
        if (dst) dst[4 * u + q] = t;
    }
}

// ---------------------------------------------------------------------------------------------
// forward, row-per-thread form of the hot configuration (float, KBCAST parameters, E/4 <= 16).  k_latent_fwd_fast
// above maps lanes to the float4 units of a row, so every row sum is a segmented shuffle reduction and every slice of
// four particles redoes the row's parameter transform: ncu round 2 counted 4.5 M warp instructions (~280 per float4 of
// latents, of which the noise is ~75) at 58 % issue utilisation -- 9.3 us for 8 MB.  Here
//   * a CTA owns 32 consecutive batch rows; their parameter-only terms (mean, std, 0.5/std^2 | probs and the log-odds
//     term; the prior's unless it is the standard one) are transformed ONCE per CTA into shared memory, and the per-row
//     constant sum_e (c - log std_e) is reduced there too;
//   * a lane owns ONE (particle, row) pair: it walks the row's E/4 units, two Philox / Box-Muller chains in flight,
//     and keeps log q and log p in registers -- no shuffles at all;
//   * the 32 rows of a particle are one contiguous 32*E-float block of z: the warp stages it in shared memory (row
//     pitch E + 4 floats: conflict-free 128-bit accesses) and writes it out with fully coalesced 128-bit stores.
// Element (k, m, e) still draws word e%4 of Philox counter (k*M*E + m*E + e)/4: the stream is identical to every other
// sampling kernel's.  Sums are re-associated (sequential over the row) against the reference's order: 1e-7 relative.
// ---------------------------------------------------------------------------------------------
constexpr int LR_WARPS = 4;
constexpr int LR_ILP = 5;  // units of a row in flight per lane

template <int FAM, bool STDP>
__global__ void __launch_bounds__(LR_WARPS * 32)
    k_latent_fwd_rows(float* __restrict__ z, float* __restrict__ logq, float* __restrict__ logp,
                      const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ pa,
                      const float* __restrict__ pb, const float* __restrict__ noise_in, int K, int M, int E4, int KS,
                      unsigned inv_e4, uint64_t seed, uint64_t offset, unsigned long long* rs,
                      unsigned char* __restrict__ zbits) {
    extern __shared__ __align__(16) float lr_smem[];
    pdl_wait();
    pdl_trigger();
    constexpr int NP = FAM == FAM_NORMAL ? (STDP ? 3 : 5) : (STDP ? 2 : 3);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int E = 4 * E4, EP = E + 4, QP = E4 + 1;
    const int m0 = (int)blockIdx.x * 32;
    const int rows = M - m0 < 32 ? M - m0 : 32;
    float* P = lr_smem;                          // [NP][32][EP]
    float* s_q = P + NP * 32 * EP;               // [32][QP] per-unit parts of the row constant of log q
    float* s_p = s_q + 32 * QP;                  // [32][QP] ... of log p
    float* stage = s_p + 32 * QP + warp * 32 * EP;  // this warp's z block [32][EP]
    const float c = normal_c<float>();
    // the stream position: the leader's load is issued now and consumed after the transform (rng_acquire_peeked)
    unsigned long long rng_base = 0ull;
    if (rs != nullptr && threadIdx.x == 0) rng_base = *reinterpret_cast<volatile unsigned long long*>(rs);
    // ---- the CTA's parameter transform, once
    for (int u = threadIdx.x; u < rows * E4; u += LR_WARPS * 32) {
        const int r = (int)(((unsigned)u * inv_e4) >> 16), j = u - r * E4;
        const size_t g = 4 * ((size_t)m0 * E4 + u);
        const float4 av = *reinterpret_cast<const float4*>(a + g);
        float4* dst = reinterpret_cast<float4*>(P + r * EP + 4 * j);
        const int PS = 32 * EP / 4;  // float4 stride between parameter arrays
        float uq, up = 0.f;
        if (FAM == FAM_NORMAL) {
            const float4 bv = *reinterpret_cast<const float4*>(b + g);
            dst[0] = av;
            dst[PS] = bv;
            dst[2 * PS] = make_float4(0.5f * lat_rcp(bv.x * bv.x), 0.5f * lat_rcp(bv.y * bv.y),
                                      0.5f * lat_rcp(bv.z * bv.z), 0.5f * lat_rcp(bv.w * bv.w));
            uq = (c - lat_log(bv.x)) + (c - lat_log(bv.y)) + (c - lat_log(bv.z)) + (c - lat_log(bv.w));
            if (!STDP) {
                float4 pm = make_float4(0.f, 0.f, 0.f, 0.f), ps = make_float4(1.f, 1.f, 1.f, 1.f);
                if (pa) pm = *reinterpret_cast<const float4*>(pa + g);
                if (pb) ps = *reinterpret_cast<const float4*>(pb + g);
                dst[3 * PS] = pm;
                dst[4 * PS] = make_float4(0.5f * lat_rcp(ps.x * ps.x), 0.5f * lat_rcp(ps.y * ps.y),
                                          0.5f * lat_rcp(ps.z * ps.z), 0.5f * lat_rcp(ps.w * ps.w));
                up = (c - lat_log(ps.x)) + (c - lat_log(ps.y)) + (c - lat_log(ps.z)) + (c - lat_log(ps.w));
            }
        } else {
            // log(p + 1e-8), log((1-p) + 1e-8) of bernoulli.py:94: l1 + z (l0 - l1) per element
            const float4 l1 = make_float4(lat_log((1.f - av.x) + 1e-8f), lat_log((1.f - av.y) + 1e-8f),
                                          lat_log((1.f - av.z) + 1e-8f), lat_log((1.f - av.w) + 1e-8f));
            dst[0] = av;
            dst[PS] = make_float4(lat_log(av.x + 1e-8f) - l1.x, lat_log(av.y + 1e-8f) - l1.y,
                                  lat_log(av.z + 1e-8f) - l1.z, lat_log(av.w + 1e-8f) - l1.w);
            uq = (l1.x + l1.y) + (l1.z + l1.w);
            if (!STDP) {
                const float4 pp = *reinterpret_cast<const float4*>(pa + g);
                const float4 h1 = make_float4(lat_log((1.f - pp.x) + 1e-8f), lat_log((1.f - pp.y) + 1e-8f),
                                              lat_log((1.f - pp.z) + 1e-8f), lat_log((1.f - pp.w) + 1e-8f));
                dst[2 * PS] = make_float4(lat_log(pp.x + 1e-8f) - h1.x, lat_log(pp.y + 1e-8f) - h1.y,
                                          lat_log(pp.z + 1e-8f) - h1.z, lat_log(pp.w + 1e-8f) - h1.w);
                up = (h1.x + h1.y) + (h1.z + h1.w);
            }
        }
        s_q[r * QP + j] = uq;
        s_p[r * QP + j] = up;
    }
    // its barrier also publishes the transform
    offset = rng_acquire_peeked(offset, rs, rng_base);
    const bool active = lane < rows;
    float cq = 0.f, cp = 0.f;
    if (active) {
        for (int j = 0; j < E4; ++j) {
            cq += s_q[lane * QP + j];
            cp += s_p[lane * QP + j];
        }
        if (STDP) cp = FAM == FAM_NORMAL ? (float)E * c : (float)E * lat_log(0.5f + 1e-8f);
    }
    const unsigned ME4 = (unsigned)M * (unsigned)E4;
    const float* prow = P + lane * EP;
    const int PSF = 32 * EP;  // float stride between parameter arrays
    for (int k = (int)blockIdx.y + KS * warp; k < K; k += KS * LR_WARPS) {  // uniform over the warp
        float accq = cq, accp = cp;
        const unsigned unit0 = (unsigned)k * ME4 + (unsigned)(m0 + lane) * (unsigned)E4;
        if (active) {
            // LR_ILP units at a time: their Philox / Box-Muller chains are independent and the kernel runs at ~11 warps
            // per SM, so the instruction-level parallelism is what hides the chains' latency
            for (int j0 = 0; j0 < E4; j0 += LR_ILP) {
                float n4[LR_ILP][4];
#pragma unroll
                for (int i = 0; i < LR_ILP; ++i) {
                    const int j = j0 + i < E4 ? j0 + i : E4 - 1;  // the tail recomputes the last unit (discarded below)
                    if (noise_in) {
                        const float4 t = *reinterpret_cast<const float4*>(noise_in + 4 * (size_t)(unit0 + j));
                        n4[i][0] = t.x; n4[i][1] = t.y; n4[i][2] = t.z; n4[i][3] = t.w;
                    } else if (FAM == FAM_NORMAL) {
                        philox_normal4((uint64_t)(unit0 + j), offset, seed, n4[i]);
                    } else {
                        philox_uniform4((uint64_t)(unit0 + j), offset, seed, n4[i]);
                    }
                }
#pragma unroll
                for (int i = 0; i < LR_ILP; ++i) {
                    const int j = j0 + i;
                    if (j >= E4) break;
                    const float4 av = *reinterpret_cast<const float4*>(prow + 4 * j);
                    float4 zv;
                    if (FAM == FAM_NORMAL) {
                        const float4 bv = *reinterpret_cast<const float4*>(prow + PSF + 4 * j);
                        const float4 h = *reinterpret_cast<const float4*>(prow + 2 * PSF + 4 * j);
                        zv = make_float4(fmaf(bv.x, n4[i][0], av.x), fmaf(bv.y, n4[i][1], av.y), fmaf(bv.z, n4[i][2], av.z),
                                         fmaf(bv.w, n4[i][3], av.w));  // normal.py:105
                        const float d0 = zv.x - av.x, d1 = zv.y - av.y, d2 = zv.z - av.z, d3 = zv.w - av.w;  // :121-124
                        accq -= (h.x * (d0 * d0) + h.y * (d1 * d1)) + (h.z * (d2 * d2) + h.w * (d3 * d3));
                        if (STDP) {
                            accp -= 0.5f * ((zv.x * zv.x + zv.y * zv.y) + (zv.z * zv.z + zv.w * zv.w));
                        } else {
                            const float4 pm = *reinterpret_cast<const float4*>(prow + 3 * PSF + 4 * j);
                            const float4 hp = *reinterpret_cast<const float4*>(prow + 4 * PSF + 4 * j);
                            const float e0 = zv.x - pm.x, e1 = zv.y - pm.y, e2 = zv.z - pm.z, e3 = zv.w - pm.w;
                            accp -= (hp.x * (e0 * e0) + hp.y * (e1 * e1)) + (hp.z * (e2 * e2) + hp.w * (e3 * e3));
                        }
                    } else {
                        const float4 l0 = *reinterpret_cast<const float4*>(prow + PSF + 4 * j);
                        zv = make_float4(n4[i][0] < av.x ? 1.f : 0.f, n4[i][1] < av.y ? 1.f : 0.f,
                                         n4[i][2] < av.z ? 1.f : 0.f, n4[i][3] < av.w ? 1.f : 0.f);  // bernoulli.py:79
                        accq += (zv.x * l0.x + zv.y * l0.y) + (zv.z * l0.z + zv.w * l0.w);
                        if (!STDP) {
                            const float4 pm = *reinterpret_cast<const float4*>(prow + 2 * PSF + 4 * j);
                            accp += (zv.x * pm.x + zv.y * pm.y) + (zv.z * pm.z + zv.w * pm.w);
                        }
                    }
                    *reinterpret_cast<float4*>(stage + lane * EP + 4 * j) = zv;
                    if (FAM == FAM_BERNOULLI && zbits)
                        zbits[unit0 + j] = (unsigned char)((zv.x != 0.f ? 1 : 0) | (zv.y != 0.f ? 2 : 0) |
                                                           (zv.z != 0.f ? 4 : 0) | (zv.w != 0.f ? 8 : 0));
                }
            }
            if (logq) logq[(size_t)k * M + m0 + lane] = accq;
            if (logp) logp[(size_t)k * M + m0 + lane] = accp;
        }
        __syncwarp();
        // the particle's 32-row block of z, coalesced
        float* zblk = z + 4 * ((size_t)k * ME4 + (size_t)m0 * E4);
        for (int u = lane; u < rows * E4; u += 32) {
            const int r = (int)(((unsigned)u * inv_e4) >> 16), j = u - r * E4;
            *reinterpret_cast<float4*>(zblk + 4 * (size_t)u) = *reinterpret_cast<const float4*>(stage + r * EP + 4 * j);
        }
        __syncwarp();
    }
}

static int g_latent_fwd_override = -1;
static bool g_latent_fwd_override_set = false;

template <int FAM>
static bool latent_fwd_rows_f32(float* z, float* logq, float* logp, const float* a, int a_mode, const float* b,
                                const float* pa, const float* pb, const float* noise_in, int64_t K, int64_t M,
                                int64_t E4, uint64_t seed, uint64_t offset, unsigned long long* rs, cudaStream_t st,
                                unsigned char* zbits) {
    // -1: by shape (below); 0: never (lane-per-unit kernel); 1: whenever the shape qualifies.  ZS_LATENT_FWD_ROWS sets
    // the process default, zs_debug_set_latent_fwd overrides it at run time (tests run both kernels on every shape).
    static const int env_choice = [] {
        const char* e = getenv("ZS_LATENT_FWD_ROWS");
        return e ? (e[0] == '0' ? 0 : 1) : -1;
    }();
    const int choice = g_latent_fwd_override >= -1 && g_latent_fwd_override_set ? g_latent_fwd_override : env_choice;
    if (choice == 0 || a_mode != ZS_KBCAST || E4 > 16 || E4 < 1 || K < 1 || M < 1 || K * M * E4 >= ((int64_t)1 << 31))
        return false;
    const int E = (int)(4 * E4), EP = E + 4, QP = (int)E4 + 1;
    const bool stdp = FAM == FAM_NORMAL ? (pa == nullptr && pb == nullptr) : pa == nullptr;
    const int np = FAM == FAM_NORMAL ? (stdp ? 3 : 5) : (stdp ? 2 : 3);
    const size_t smem = (size_t)(np * 32 * EP + 2 * 32 * QP + LR_WARPS * 32 * EP) * sizeof(float);
    // one particle per warp unless that takes more CTAs than the machine holds a few times over
    const int64_t tiles = (M + 31) / 32;
    int64_t per_warp = 1;
    while (tiles * ((K + LR_WARPS * per_warp - 1) / (LR_WARPS * per_warp)) > (int64_t)sm_count() * 16 && per_warp < K)
        per_warp *= 2;
    int64_t KS = (K + LR_WARPS * per_warp - 1) / (LR_WARPS * per_warp);
    if (KS > 65535 || tiles >= (int64_t)2147483647) return false;
    // Measured with tools/step_breakdown.py at K = 50, Z = 40 (profiles/r2_notes.md): the row form executes a third
    // fewer instructions but runs few, fat warps, so it wins once the grid is several waves deep (B = 4096: 20.5
    // against 27.1 us, B = 8192: 35.3 against 65.5 us), ties at B = 1024 (416 CTAs, 2.8 per SM) and loses below
    // (B = 128: 5.4 against 3.6 us).  By default it takes grids of at least six CTAs per SM.
    if (choice < 0 && tiles * KS < (int64_t)sm_count() * 6) return false;
    const unsigned inv = (unsigned)((65536 + E4 - 1) / E4);
    auto kern = stdp ? k_latent_fwd_rows<FAM, true> : k_latent_fwd_rows<FAM, false>;
    if (cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        (void)cudaGetLastError();
        return false;
    }
    launch_pdl(PDL_LATENT_FWD, kern, dim3((unsigned)tiles, (unsigned)KS), dim3(LR_WARPS * 32), smem, st, z, logq, logp, a,
               b, pa, pb, noise_in, (int)K, (int)M, (int)E4, (int)KS, inv, seed, offset, rs, zbits);
    return true;
}

// float / KBCAST / 32-bit indexable shapes go to k_latent_fwd_fast; returns false when the shape does not qualify
template <typename T, int FAM>
static bool launch_latent_fwd_fast(dim3 grid, T* z, T* logq, T* logp, const T* a, int a_mode, const T* b, const T* pa,
                                   const T* pb, const T* noise_in, int64_t K, int64_t M, int64_t E4, int RW, int64_t KS,
                                   uint64_t seed, uint64_t offset, unsigned long long* rs, cudaStream_t st,
                                   unsigned char* zbits) {
    if constexpr (std::is_same<T, float>::value) {
        if (a_mode != ZS_KBCAST || K * M * E4 >= ((int64_t)1 << 31) || K * M >= ((int64_t)1 << 31)) return false;
        if (latent_fwd_rows_f32<FAM>(z, logq, logp, a, a_mode, b, pa, pb, noise_in, K, M, E4, seed, offset, rs, st,
                                     zbits))
            return true;
        const unsigned inv = (unsigned)((65536 + E4 - 1) / E4);
        const bool stdp = FAM == FAM_NORMAL ? (pa == nullptr && pb == nullptr) : pa == nullptr;
        launch_pdl(PDL_LATENT_FWD, stdp ? k_latent_fwd_fast<FAM, true> : k_latent_fwd_fast<FAM, false>, grid,
                   dim3(LF_WARPS * 32), 0, st, z, logq, logp, a, b, pa, pb, noise_in, (int)K, (int)M, (int)E4, RW,
                   (int)KS, inv, seed, offset, rs, zbits);
        return true;
    }
    return false;
}

template <typename T, int FAM>
static int launch_latent_fwd(T* z, T* logq, T* logp, const T* a, int a_mode, const T* b, int b_mode, const T* pa,
                             const T* pb, const T* noise_in, int64_t K, int64_t M, int64_t E, uint64_t seed,
                             uint64_t offset, unsigned long long* rs, cudaStream_t st, unsigned char* zbits = nullptr) {
    if (noise_in) rs = nullptr;  // injected noise: no draw, the stream position stays
    const int64_t E4 = E >> 2;
    if (E4 <= 32 && K < ((int64_t)1 << 30)) {
        const int RW = (int)(32 / E4);
        const int64_t row_warps = (M + RW - 1) / RW;
        const int64_t gx = (row_warps + LF_WARPS - 1) / LF_WARPS;
        // k-slices: two particles in flight per thread (two Philox / Box-Muller chains), and as many pairs per
        // thread as it takes for the whole grid to be resident at once (8 CTAs of 4 warps per SM at 60 registers):
        // a 1.2-wave grid leaves the machine a quarter full for the length of its second wave.  The parameter
        // terms a slice recomputes are SFU ops (lat_log / lat_rcp), so slices are cheap.  Config 2 (K = 50,
        // M = 1024, Z = 40): 86 CTAs x 13 slices of 4 particles = 1118 CTAs on 148 x 8 slots.
        const int64_t resident = (int64_t)sm_count() * 8;
        int64_t trips = K < 2 ? 1 : 2;
        while (gx * ((K + trips - 1) / trips) > resident && trips < K) trips += 2;
        int64_t KS = (K + trips - 1) / trips;
        if (KS > 65535) KS = 65535;
        if (KS < 1) KS = 1;
        ZS_REQUIRE(gx < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);
        dim3 grid((unsigned)gx, (unsigned)KS);
        if (launch_latent_fwd_fast<T, FAM>(grid, z, logq, logp, a, a_mode, b, pa, pb, noise_in, K, M, E4, RW, KS, seed,
                                           offset, rs, st, zbits)) {
            ZS_LAUNCH_CHECK("k_latent_fwd_fast");
            return ZS_OK;
        }
        if (zbits) {
            set_last_error_msg("the packed sample (zbits) is produced by the float32 / KBCAST forward kernels only");
            return ZS_ERR_UNSUPPORTED;
        }
        k_latent_fwd_packed<T, FAM><<<grid, LF_WARPS * 32, 0, st>>>(z, logq, logp, a, a_mode, b, pa, pb, noise_in, (int)K, M,
                                                                    (int)E4, RW, (int)KS, seed, offset, rs);
        ZS_LAUNCH_CHECK("k_latent_fwd_packed");
        return ZS_OK;
    }
    if (zbits) {
        set_last_error_msg("the packed sample (zbits) is produced by the float32 / KBCAST forward kernels only");
        return ZS_ERR_UNSUPPORTED;
    }
    // k-slices per batch row: enough groups to fill the machine, each slice reusing its parameters
#define ZS_LATENT_FWD(G)                                                                                          \
    {                                                                                                             \
        int64_t KS = (int64_t)sm_count() * 2048 / (M * G > 0 ? M * G : 1);                                        \
        if (KS < 1) KS = 1;                                                                                       \
        if (KS > K) KS = K;                                                                                       \
        if (KS > 16) KS = 16;                                                                                     \
        const int64_t groups = M * KS;                                                                            \
        const int64_t grid = (groups * G + 255) / 256;                                                            \
        ZS_REQUIRE(grid < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);                                               \
        k_latent_fwd<T, FAM, G><<<(unsigned)grid, 256, 0, st>>>(z, logq, logp, a, a_mode, b, b_mode, pa, pb,      \
                                                                noise_in, K, M, E, (int)KS, seed, offset, rs);    \
    }
    if (E4 <= 4) ZS_LATENT_FWD(4)
    else if (E4 <= 8) ZS_LATENT_FWD(8)
    else if (E4 <= 16) ZS_LATENT_FWD(16)
    else ZS_LATENT_FWD(32)
#undef ZS_LATENT_FWD
    ZS_LAUNCH_CHECK("k_latent_fwd");
    return ZS_OK;
}

static int latent_args_ok(const void* a, int a_mode, const void* b, int b_mode, int fam, int64_t E,
                          std::initializer_list<const void*> ptrs) {
    if (E % 4 != 0) {
        set_last_error_msg("latent kernels need E % 4 == 0");
        return ZS_ERR_UNSUPPORTED;
    }
    if (!(a_mode == ZS_FULL || a_mode == ZS_KBCAST) || (fam == FAM_NORMAL && b_mode != a_mode)) {
        set_last_error_msg("latent kernels need both variational parameters FULL or both KBCAST");
        return ZS_ERR_UNSUPPORTED;
    }
    for (const void* p : ptrs)
        if (!aligned16(p)) {
            set_last_error_msg("latent kernels need 16-byte aligned tensors");
            return ZS_ERR_ALIGN;
        }
    (void)a;
    (void)b;
    return ZS_OK;
}

// ---------------------------------------------------------------------------------------------
// backward, the hot configuration (float, KBCAST parameters, 32-bit indexable).  The generic kernel above mirrors
// autograd term by term (~50 floating-point instructions per element, 4.5 M warp instructions at config 2) and was
// latency- AND issue-bound at 11 us for 17 MB.  Algebra first: with z = mean + std*eps and d = z - mean,
//     d log q / d mean  through the density (+g prec d) and through the sample (-g prec d) cancel exactly,
//     d log q / d std   = -g/std  after the same cancellation of the (g d^2 prec / std) pair,
// so for a reparameterised node, with t = dz_up + d(log p)/dz the gradient reaching the sample from outside,
//     dmean = sum_k t          dstd = sum_k (t * d - g_q) / std
// and for a non-reparameterised one  dmean = sum_k g_q prec d,  dstd = sum_k g_q (d^2 prec - 1) / std.
// The reference computes the cancelling pairs and adds them up in float32; this form has no cancellation (it is the
// closer of the two to the float64 reference run) and ~8 instructions per element.  Four particles per thread, all
// eight 128-bit loads issued before the first use.
// ---------------------------------------------------------------------------------------------
constexpr int LBF_U = 4;  // particles in flight per thread (default)

// LBF_U > 4: the one-wave block shape of config 2 (8 x 8 threads, 17 warps per SM) walked K = 50 particles in TWO
// dependent rounds of loads (4 + 3 per thread) and was latency-bound on them (ncu round 2: long_scoreboard 10 of 13
// stall cycles per issue, 2 TB/s).  With ceil(K / slices) <= 8 particles per thread ALL loads of the thread are issued
// before the first use -- one memory round trip per CTA -- at ~100 registers, which 17 warps per SM can afford.
template <int FAM, bool STDP, int LBF_U>
__global__ void __launch_bounds__(LB_X_MAX* LB_Y_MAX, LBF_U > 4 ? 2 : 4)
    k_latent_bwd_fast(float* __restrict__ da, float* __restrict__ db, const float* __restrict__ gq,
                      const float* __restrict__ gp, const float* __restrict__ dz_up, const float* __restrict__ z,
                      const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ pa,
                      const float* __restrict__ pb, int reparam, int K, int M, int E,
                      const unsigned char* __restrict__ zbits) {
    pdl_wait();
    pdl_trigger();
    const int LBX = blockDim.x, LBY = blockDim.y;
    const unsigned ME4 = ((unsigned)M * (unsigned)E) >> 2;
    const unsigned u = blockIdx.x * LBX + threadIdx.x;
    const bool valid = u < ME4;
    float4 sa = make_float4(0.f, 0.f, 0.f, 0.f), sb = sa;
    if (valid) {
        const unsigned m = (4u * u) / (unsigned)E;
        const float4 av = *reinterpret_cast<const float4*>(a + 4 * (size_t)u);
        float4 r0, r1 = make_float4(0.f, 0.f, 0.f, 0.f), pm = r1, pprec = make_float4(1.f, 1.f, 1.f, 1.f);
        if (FAM == FAM_NORMAL) {
            const float4 sd = *reinterpret_cast<const float4*>(b + 4 * (size_t)u);
            r0 = make_float4(lat_rcp(sd.x), lat_rcp(sd.y), lat_rcp(sd.z), lat_rcp(sd.w));  // 1/std
            if (!STDP) {
                if (pa) pm = *reinterpret_cast<const float4*>(pa + 4 * (size_t)u);
                if (pb) {
                    const float4 ps = *reinterpret_cast<const float4*>(pb + 4 * (size_t)u);
                    pprec = make_float4(lat_rcp(ps.x * ps.x), lat_rcp(ps.y * ps.y), lat_rcp(ps.z * ps.z),
                                        lat_rcp(ps.w * ps.w));
                }
            }
        } else {
            // bernoulli.py:94's autograd wrt probs: g (z / (p + eps) - (1 - z) / ((1 - p) + eps))
            r0 = make_float4(lat_rcp(av.x + 1e-8f), lat_rcp(av.y + 1e-8f), lat_rcp(av.z + 1e-8f), lat_rcp(av.w + 1e-8f));
            r1 = make_float4(lat_rcp((1.f - av.x) + 1e-8f), lat_rcp((1.f - av.y) + 1e-8f), lat_rcp((1.f - av.z) + 1e-8f),
                             lat_rcp((1.f - av.w) + 1e-8f));
        }
        const bool path = reparam != 0 && FAM == FAM_NORMAL;
        const bool has_du = path && dz_up != nullptr, has_gp = path && gp != nullptr;
        for (int k0 = threadIdx.y; k0 < K; k0 += LBF_U * LBY) {
            float g_q[LBF_U], g_p[LBF_U];
            float4 zv[LBF_U], du[LBF_U];
#pragma unroll
            for (int i = 0; i < LBF_U; ++i) {
                const int k = k0 + i * LBY;
                const unsigned kc = (unsigned)(k < K ? k : k0);  // always in bounds
                const unsigned r = kc * (unsigned)M + m;
                const size_t fe = 4 * ((size_t)kc * ME4 + u);
                g_q[i] = gq ? __ldg(gq + r) : 0.f;
                g_p[i] = has_gp ? __ldg(gp + r) : 0.f;
                if (FAM == FAM_BERNOULLI && zbits != nullptr) {
                    // the forward's packed copy of the sample (one byte per float4 unit): 1/16 of the bytes, which
                    // matters behind the fused kernel, whose write-back is still draining when this kernel reads
                    const unsigned bb = zbits[(size_t)kc * ME4 + u];
                    zv[i] = make_float4((bb & 1u) ? 1.f : 0.f, (bb & 2u) ? 1.f : 0.f, (bb & 4u) ? 1.f : 0.f,
                                        (bb & 8u) ? 1.f : 0.f);
                } else {
                    zv[i] = *reinterpret_cast<const float4*>(z + fe);
                }
                du[i] = has_du ? *reinterpret_cast<const float4*>(dz_up + fe) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
#pragma unroll
            for (int i = 0; i < LBF_U; ++i) {
                if (k0 + i * LBY >= K) break;
                const float g = g_q[i], h = g_p[i];
                if (FAM == FAM_NORMAL) {
                    const float d0 = zv[i].x - av.x, d1 = zv[i].y - av.y, d2 = zv[i].z - av.z, d3 = zv[i].w - av.w;
                    if (path) {
                        float t0 = du[i].x, t1 = du[i].y, t2 = du[i].z, t3 = du[i].w;
                        if (STDP) {  // d/dz of c - z^2/2
                            t0 = fmaf(-h, zv[i].x, t0); t1 = fmaf(-h, zv[i].y, t1);
                            t2 = fmaf(-h, zv[i].z, t2); t3 = fmaf(-h, zv[i].w, t3);
                        } else {
                            t0 = fmaf(-h * pprec.x, zv[i].x - pm.x, t0); t1 = fmaf(-h * pprec.y, zv[i].y - pm.y, t1);
                            t2 = fmaf(-h * pprec.z, zv[i].z - pm.z, t2); t3 = fmaf(-h * pprec.w, zv[i].w - pm.w, t3);
                        }
                        sa.x += t0; sa.y += t1; sa.z += t2; sa.w += t3;
                        sb.x += fmaf(t0, d0, -g); sb.y += fmaf(t1, d1, -g);
                        sb.z += fmaf(t2, d2, -g); sb.w += fmaf(t3, d3, -g);
                    } else {  // score-function estimators: the sample carries no gradient
                        const float e0 = d0 * r0.x, e1 = d1 * r0.y, e2 = d2 * r0.z, e3 = d3 * r0.w;  // eps
                        sa.x += g * e0; sa.y += g * e1; sa.z += g * e2; sa.w += g * e3;   // x 1/std below
                        sb.x += g * fmaf(e0, e0, -1.f); sb.y += g * fmaf(e1, e1, -1.f);
                        sb.z += g * fmaf(e2, e2, -1.f); sb.w += g * fmaf(e3, e3, -1.f);
                    }
                } else {
                    sa.x += g * (zv[i].x != 0.f ? r0.x : -r1.x); sa.y += g * (zv[i].y != 0.f ? r0.y : -r1.y);
                    sa.z += g * (zv[i].z != 0.f ? r0.z : -r1.z); sa.w += g * (zv[i].w != 0.f ? r0.w : -r1.w);
                }
            }
        }
        if (FAM == FAM_NORMAL) {  // the common 1/std factor, once
            sb.x *= r0.x; sb.y *= r0.y; sb.z *= r0.z; sb.w *= r0.w;
            if (!path) { sa.x *= r0.x; sa.y *= r0.y; sa.z *= r0.z; sa.w *= r0.w; }
        }
    }
    __shared__ float red[2][LB_Y_MAX][LB_X_MAX][4];
    red[0][threadIdx.y][threadIdx.x][0] = sa.x; red[0][threadIdx.y][threadIdx.x][1] = sa.y;
    red[0][threadIdx.y][threadIdx.x][2] = sa.z; red[0][threadIdx.y][threadIdx.x][3] = sa.w;
    red[1][threadIdx.y][threadIdx.x][0] = sb.x; red[1][threadIdx.y][threadIdx.x][1] = sb.y;
    red[1][threadIdx.y][threadIdx.x][2] = sb.z; red[1][threadIdx.y][threadIdx.x][3] = sb.w;
    __syncthreads();
    // fixed-order sum over the slices: thread (x, y < 8) adds up component (y & 3) of array (y >> 2)
    if (threadIdx.y < 8 && valid) {
        const int arr = threadIdx.y >> 2, q = threadIdx.y & 3;
        float t = 0.f;
        for (int sl = 0; sl < LBY; ++sl) t += red[arr][sl][threadIdx.x][q];
        float* dst = arr == 0 ? da : (FAM == FAM_NORMAL ? db : nullptr);
        if (dst) dst[4 * (size_t)u + q] = t;
    }
}

// float / KBCAST / 32-bit indexable shapes go to k_latent_bwd_fast; returns false when the shape does not qualify
template <int FAM>
static bool launch_latent_bwd_fast(void* da, void* db, const void* gq, const void* gp, const void* dz_up, const void* z,
                                   const void* a, int a_mode, const void* b, const void* pa, const void* pb, int reparam,
                                   int64_t K, int64_t M, int64_t E, cudaStream_t st, const void* zbits) {
    if (a_mode != ZS_KBCAST || K * M * E >= ((int64_t)1 << 31) || da == nullptr || (FAM == FAM_NORMAL && db == nullptr))
        return false;
    const int64_t ME4 = (M * E) >> 2;
    const int lbx = LB_X_MAX;
    int lby = (int)((K + LBF_U - 1) / LBF_U);
    if (lby > LB_Y_MAX) lby = LB_Y_MAX;
    if (lby < 8) lby = 8;  // the epilogue's eight (array, component) sums are taken by slices 0..7
    const unsigned grid = (unsigned)((ME4 + lbx - 1) / lbx);
    // Wave quantisation: at 64 registers an SM holds 32 warps.  A grid slightly larger than what is resident at once
    // (config 2: 1280 CTAs of 4 warps on 148 x 8 slots, "1.08 waves") runs its last few CTAs alone and doubles the
    // kernel's duration (ncu round 2: SMs active 52 % of 9.9 us).  Halve the slices (each thread then walks twice
    // as many particles, still four at a time) until the grid is resident in one go.
    {
        const int64_t warp_slots = (int64_t)sm_count() * 32;
        while (lby > 8 && (int64_t)grid * ((lbx * lby + 31) / 32) > warp_slots) lby = (lby + 1) / 2 < 8 ? 8 : (lby + 1) / 2;
    }
    dim3 block(lbx, lby);
    const bool stdp = pa == nullptr && pb == nullptr;
    auto kern = stdp ? k_latent_bwd_fast<FAM, true, LBF_U> : k_latent_bwd_fast<FAM, false, LBF_U>;
    // every particle of a thread in flight at once where that takes at most 8 (and the CTAs stay small enough for the
    // register budget: 2 x 256 threads per SM are guaranteed, the one-wave shape needs 17 warps)
    const int per_thread = (int)((K + lby - 1) / lby);
    static const bool all_in_flight = [] {  // developer knob: ZS_LATENT_BWD_DEEP=0 keeps four particles in flight
        const char* e = getenv("ZS_LATENT_BWD_DEEP");
        return !(e && e[0] == '0');
    }();
    if (lbx * lby <= 128 && all_in_flight) {
#define ZS_LBF_PICK(U) \
    if (per_thread == (U)) kern = stdp ? k_latent_bwd_fast<FAM, true, U> : k_latent_bwd_fast<FAM, false, U>
        ZS_LBF_PICK(5);
        ZS_LBF_PICK(6);
        ZS_LBF_PICK(7);
        ZS_LBF_PICK(8);
#undef ZS_LBF_PICK
    }
    launch_pdl(PDL_LATENT_BWD, kern, dim3(grid), block, 0, st, (float*)da, (float*)db, (const float*)gq, (const float*)gp,
               (const float*)dz_up, (const float*)z, (const float*)a, (const float*)b, (const float*)pa,
               (const float*)pb, reparam, (int)K, (int)M, (int)E, (const unsigned char*)zbits);
    return true;
}

template <typename T, int FAM>
static int launch_latent_bwd(void* da, void* db, const void* gq, const void* gp, const void* dz_up, const void* z,
                             const void* a, int a_mode, const void* b, int b_mode, const void* pa, const void* pb,
                             int reparam, int64_t K, int64_t M, int64_t E, zs_stream_t stream,
                             const void* zbits = nullptr) {
    if (std::is_same<T, float>::value && launch_latent_bwd_fast<FAM>(da, db, gq, gp, dz_up, z, a, a_mode, b, pa, pb,
                                                                     reparam, K, M, E, as_stream(stream), zbits)) {
        ZS_LAUNCH_CHECK("k_latent_bwd_fast");
        return ZS_OK;
    }
    const int64_t ME4 = (M * E) >> 2;
    // blockDim.x float4 units of [M,E] (8 = one 128-byte line per particle row; 4 when that leaves fewer than ~16
    // CTAs per SM: the grid is a few waves deep, so small CTAs keep the last wave's imbalance small)
    static const int forced_x = [] {
        const char* e = getenv("ZS_LATENT_BWD_X");
        return e ? atoi(e) : 0;
    }();
    int lbx = (ME4 / LB_X_MAX >= (int64_t)sm_count() * 16) ? LB_X_MAX : 4;
    if (forced_x == 4 || forced_x == 8) lbx = forced_x;
    const int64_t grid = (ME4 + lbx - 1) / lbx;
    ZS_REQUIRE(grid < (int64_t)2147483647, ZS_ERR_UNSUPPORTED);
    int lby = (int)((K + 1) / 2);  // two particles per thread
    if (lby > LB_Y_MAX) lby = LB_Y_MAX;
    if (lby < 8) lby = 8;          // the epilogue's eight (array, component) sums are taken by slices 0..7
    dim3 block(lbx, lby);
    const bool stdp = pa == nullptr && pb == nullptr;
    auto kern = stdp ? k_latent_bwd<T, FAM, true> : k_latent_bwd<T, FAM, false>;
    kern<<<(unsigned)grid, block, 0, as_stream(stream)>>>(
        (T*)da, (T*)db, (const T*)gq, (const T*)gp, (const T*)dz_up, (const T*)z, (const T*)a, a_mode, (const T*)b,
        b_mode, (const T*)pa, (const T*)pb, reparam, K, M, E);
    ZS_LAUNCH_CHECK("k_latent_bwd");
    return ZS_OK;
}

}  // namespace zs

using namespace zs;

extern "C" int zs_debug_set_latent_fwd(int impl) {
    ZS_REQUIRE(impl >= -1 && impl <= 1, ZS_ERR_ARG);
    zs::g_latent_fwd_override = impl;
    zs::g_latent_fwd_override_set = true;
    return ZS_OK;
}

extern "C" {

int zs_normal_latent_fwd(int dtype, void* z, void* logq, void* logp, const void* mean, int mean_mode, const void* std,
                         int std_mode, const void* prior_mean, const void* prior_std, const void* eps_in, int64_t K,
                         int64_t M, int64_t E, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream) {
    ZS_REQUIRE(z && mean && std && K >= 0 && M >= 0 && E >= 1, ZS_ERR_ARG);
    int rc = latent_args_ok(mean, mean_mode, std, std_mode, FAM_NORMAL, E, {z, mean, std, prior_mean, prior_std, eps_in});
    if (rc != ZS_OK) return rc;
    if (K * M == 0) return ZS_OK;
    ZS_DTYPE_SWITCH(dtype, {
        return launch_latent_fwd<T, FAM_NORMAL>((T*)z, (T*)logq, (T*)logp, (const T*)mean, mean_mode, (const T*)std,
                                                std_mode, (const T*)prior_mean, (const T*)prior_std, (const T*)eps_in,
                                                K, M, E, seed, offset, (unsigned long long*)rng_state,
                                                as_stream(stream));
    })
}

int zs_bernoulli_latent_fwd(int dtype, void* z, void* logq, void* logp, const void* probs, int probs_mode,
                            const void* prior_probs, const void* u_in, int64_t K, int64_t M, int64_t E, uint64_t seed,
                            uint64_t offset, void* rng_state, void* zbits, zs_stream_t stream) {
    ZS_REQUIRE(z && probs && K >= 0 && M >= 0 && E >= 1, ZS_ERR_ARG);
    ZS_REQUIRE(zbits == nullptr || dtype == ZS_F32, ZS_ERR_UNSUPPORTED);
    int rc = latent_args_ok(probs, probs_mode, nullptr, probs_mode, FAM_BERNOULLI, E, {z, probs, prior_probs, u_in});
    if (rc != ZS_OK) return rc;
    if (K * M == 0) return ZS_OK;
    ZS_DTYPE_SWITCH(dtype, {
        return launch_latent_fwd<T, FAM_BERNOULLI>((T*)z, (T*)logq, (T*)logp, (const T*)probs, probs_mode, nullptr,
                                                   probs_mode, (const T*)prior_probs, nullptr, (const T*)u_in, K, M, E,
                                                   seed, offset, (unsigned long long*)rng_state, as_stream(stream),
                                                   (unsigned char*)zbits);
    })
}

int zs_normal_latent_bwd(int dtype, void* dmean, void* dstd, const void* dlogq, const void* dlogp, const void* dz_up,
                         const void* z, const void* mean, int mean_mode, const void* std, int std_mode,
                         const void* prior_mean, const void* prior_std, int reparameterized, int64_t K, int64_t M,
                         int64_t E, zs_stream_t stream) {
    ZS_REQUIRE(z && mean && std && K >= 0 && M >= 0 && E >= 1, ZS_ERR_ARG);
    int rc = latent_args_ok(mean, mean_mode, std, std_mode, FAM_NORMAL, E,
                            {dmean, dstd, dz_up, z, mean, std, prior_mean, prior_std});
    if (rc != ZS_OK) return rc;
    if (K * M == 0 || (!dmean && !dstd)) return ZS_OK;
    ZS_DTYPE_SWITCH(dtype, {
        return launch_latent_bwd<T, FAM_NORMAL>(dmean, dstd, dlogq, dlogp, dz_up, z, mean, mean_mode, std, std_mode,
                                                prior_mean, prior_std, reparameterized, K, M, E, stream);
    })
}

int zs_bernoulli_latent_bwd(int dtype, void* dprobs, const void* dlogq, const void* z, const void* probs,
                            int probs_mode, int64_t K, int64_t M, int64_t E, const void* zbits, zs_stream_t stream) {
    ZS_REQUIRE(dprobs && dlogq && z && probs && K >= 0 && M >= 0 && E >= 1, ZS_ERR_ARG);
    int rc = latent_args_ok(probs, probs_mode, nullptr, probs_mode, FAM_BERNOULLI, E, {dprobs, z, probs});
    if (rc != ZS_OK) return rc;
    if (K * M == 0) return ZS_OK;
    ZS_DTYPE_SWITCH(dtype, {
        return launch_latent_bwd<T, FAM_BERNOULLI>(dprobs, nullptr, dlogq, nullptr, nullptr, z, probs, probs_mode,
                                                   nullptr, probs_mode, nullptr, nullptr, 0, K, M, E, stream, zbits);
    })
}

}  // extern "C"
