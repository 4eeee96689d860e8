// Fused resident-column kernel: Bernoulli likelihood log-pmf + importance-weighted objective
// (SGVB or VIMCO), forward AND backward, one launch, probs read from HBM once.  The fixed-geometry box kernel also
// has a Poisson-likelihood instantiation (k_iw_poisson_boxf: rates [K,B,X], counts x [B,X]).
//
// Replaces, for a Bernoulli likelihood node under ImportanceWeightedObjective (reference file:line):
//   Bernoulli._log_prob            zhusuan/distributions/bernoulli.py:84-95   (fwd + autograd bwd)
//   StochasticTensor.log_prob      zhusuan/framework/stochastic_tensor.py:160-181 (event sum)
//   ImportanceWeightedObjective.log_joint / sgvb / vimco
//                                  zhusuan/variational/importance_weighted_objective.py:66-77,102-191
//
// Three kernels live in this file; zs_iw_bernoulli_fused picks box -> generic box -> ring
// (DESIGN.md 3.1 has the measurements behind each step; the two round-1 predecessors -- whole column resident
// without prefetch, 123 us, and re-read-from-L2, 95 us -- were removed):
//   k_iw_bernoulli_ring    (ring) persistent warp-specialised CTA, per-warp rings of 1-D bulk row copies  66.5 us
//   k_iw_bernoulli_box     (boxg) column resident between its two passes, 3-D TENSOR bulk copies         69.8 us
//   k_iw_bernoulli_boxf    (box)  the same with compile-time box geometry, signed-argument x staging,
//                                 optional in-place sigmoid for logits                              62-64 us
// All of them: one persistent CTA per SM walks batch columns b; for a column
//   phase A  log-pmf of the K rows probs[k, b, :] against x[b, :]                         (warp shuffle sums)
//   sync     one named barrier; an objective warp forms log-weights, weights / VIMCO signal, cost, d/dlogp, d/dlogq
//   phase B  dprobs = g_k * (x/(p+eps) - (1-x)/((1-p)+eps)) -> HBM
// HBM traffic per particle-sample: 4X read + 4X write (+ [K,B] scalars) instead of 8X + 4X for the
// two-pass form; the unfused entry points remain as the general fallback.  The host-buffer step
// (zs_iw_step_host*) at the end of the file pipelines the same kernels over column chunks.
#include <stdio.h>
#include <stdlib.h>

#include <cuda.h>  // CUtensorMap and its enums only: the encoder is fetched at run time, libcuda is not linked

#include <initializer_list>
#include <new>

#include "zs_common.cuh"

namespace zs {

// launch flags of the fused kernels (kernel parameter `flags`)
constexpr int FUSED_ACCUMULATE = 1;   // cost[b] += cost_b (running sum over launches) instead of cost[b] = cost_b
constexpr int FUSED_EARLY_ISSUE = 2;  // ring kernel dev knob: first bulk copies before the first staging
constexpr int FUSED_COST_SCALED = 4;  // cost[b] = cost_b * grad_scale: sum_b cost[b] is the mean objective

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 128-bit shared-memory load.  Written as asm because the compiler otherwise scalarises the float4 into
// four LDS.32 whose lane stride of 16 B is a 4-way bank conflict (profiles/r1_notes.md).  volatile keeps
// it ordered after the mbarrier wait that publishes the slot.
__device__ __forceinline__ float4 lds128(const float4* p) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "r"(smem_u32(p)));
    return r;
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "ZS_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra ZS_DONE;\n"
        "bra ZS_WAIT;\n"
        "ZS_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D bulk async copy global -> shared, completion counted on an mbarrier (TMA engine, UBLKCP)
__device__ __forceinline__ void bulk_load(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void stg_hint(float* p, const float4& v, uint64_t) {
    asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}

// log-pmf contribution of 4 elements (log2 units) / their dprobs; binary x needs one SFU op per element
template <bool BINARY>
__device__ __forceinline__ float lpmf4(const float4& p, const float4& xx, float& mn) {
    if (BINARY) {
        float a, b, acc;
        a = p.x + 1e-8f; b = (1.0f - p.x) + 1e-8f; mn = fminf(mn, fminf(a, b)); acc = fast_log2(xx.x == 1.f ? a : b);
        a = p.y + 1e-8f; b = (1.0f - p.y) + 1e-8f; mn = fminf(mn, fminf(a, b)); acc += fast_log2(xx.y == 1.f ? a : b);
        a = p.z + 1e-8f; b = (1.0f - p.z) + 1e-8f; mn = fminf(mn, fminf(a, b)); acc += fast_log2(xx.z == 1.f ? a : b);
        a = p.w + 1e-8f; b = (1.0f - p.w) + 1e-8f; mn = fminf(mn, fminf(a, b)); acc += fast_log2(xx.w == 1.f ? a : b);
        return acc;
    }
    float acc = xx.x * fast_log2(p.x + 1e-8f) + (1.0f - xx.x) * fast_log2((1.0f - p.x) + 1e-8f);
    acc += xx.y * fast_log2(p.y + 1e-8f) + (1.0f - xx.y) * fast_log2((1.0f - p.y) + 1e-8f);
    acc += xx.z * fast_log2(p.z + 1e-8f) + (1.0f - xx.z) * fast_log2((1.0f - p.z) + 1e-8f);
    acc += xx.w * fast_log2(p.w + 1e-8f) + (1.0f - xx.w) * fast_log2((1.0f - p.w) + 1e-8f);
    return acc;
}
template <bool BINARY>
__device__ __forceinline__ float4 dprobs4(const float4& p, const float4& xx, float g) {
    float4 o;
    if (BINARY) {
        const float ng = -g;
        o.x = (xx.x == 1.f ? g : ng) * fast_rcp(xx.x == 1.f ? p.x + 1e-8f : (1.0f - p.x) + 1e-8f);
        o.y = (xx.y == 1.f ? g : ng) * fast_rcp(xx.y == 1.f ? p.y + 1e-8f : (1.0f - p.y) + 1e-8f);
        o.z = (xx.z == 1.f ? g : ng) * fast_rcp(xx.z == 1.f ? p.z + 1e-8f : (1.0f - p.z) + 1e-8f);
        o.w = (xx.w == 1.f ? g : ng) * fast_rcp(xx.w == 1.f ? p.w + 1e-8f : (1.0f - p.w) + 1e-8f);
    } else {
        o.x = (g * xx.x) * fast_rcp(p.x + 1e-8f) - (g * (1.0f - xx.x)) * fast_rcp((1.0f - p.x) + 1e-8f);
        o.y = (g * xx.y) * fast_rcp(p.y + 1e-8f) - (g * (1.0f - xx.y)) * fast_rcp((1.0f - p.y) + 1e-8f);
        o.z = (g * xx.z) * fast_rcp(p.z + 1e-8f) - (g * (1.0f - xx.z)) * fast_rcp((1.0f - p.z) + 1e-8f);
        o.w = (g * xx.w) * fast_rcp(p.w + 1e-8f) - (g * (1.0f - xx.w)) * fast_rcp((1.0f - p.w) + 1e-8f);
    }
    return o;
}

// Objective warp: turns the K log-weights of a column into cost, dlogp, dlogq (global) — off the
// critical path of the row warps.  Same math as k_iw_objective; reciprocal instead of IEEE division.
template <int EST>
__device__ __forceinline__ float column_objective(int lane, int K, int64_t B, int64_t b, const float* s_lpx,
                                               const float* s_other, const float* s_lq, double* s_xw, float gscale,
                                               float* __restrict__ cost, float* __restrict__ dlogp,
                                               float* __restrict__ dlogq, float* __restrict__ logpx_out,
                                               int flags = 0) {
    const bool accumulate = (flags & FUSED_ACCUMULATE) != 0;
    const float cscale = (flags & FUSED_COST_SCALED) ? gscale : 1.0f;
    // running-sum mode: the old value is requested first so its latency hides behind the objective's arithmetic
    const float prev_cost = (accumulate && lane == 0 && cost) ? cost[b] : 0.f;
    const unsigned FULL = 0xffffffffu;
    // log-weights in double; max in float (any value within an ulp of the max stabilises exp)
    float mf = -INFINITY;
    for (int k = lane; k < K; k += 32) {
        double xv = ((double)s_lpx[k] - (double)s_lq[k]) + (double)s_other[k];
        s_xw[k] = xv;
        mf = fmaxf(mf, (float)xv);
    }
    mf = warp_max(mf);
    const double m1 = (double)mf;
    float S = 0.f;
    double sumd = 0.0;
    for (int k = lane; k < K; k += 32) {
        const double d = s_xw[k] - m1;
        S += expf((float)d);
        if (EST == ZS_EST_VIMCO) sumd += d;
    }
    S = warp_sum(S);
    const float invS = fast_rcp(S) * (2.0f - S * fast_rcp(S));  // one Newton step: ~1 ulp
    float gap = 0.f, S2 = 0.f;  // gap = m1 - (second max), S2 = sum_{k != argmax} exp(x_k - second max)
    int i1 = -1;
    if (EST == ZS_EST_VIMCO) {
        sumd = warp_sum(sumd);
        // arg-max (smallest index among ties) and second max, needed only for the arg-max row
        double best = -INFINITY;
        for (int k = lane; k < K; k += 32)
            if (s_xw[k] > best) { best = s_xw[k]; i1 = k; }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            double ob = __shfl_xor_sync(FULL, best, o);
            int oi = __shfl_xor_sync(FULL, i1, o);
            if (oi >= 0 && (i1 < 0 || ob > best || (ob == best && oi < i1))) { best = ob; i1 = oi; }
        }
        double m2 = -INFINITY;
        for (int k = lane; k < K; k += 32)
            if (k != i1) m2 = fmax(m2, s_xw[k]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) m2 = fmax(m2, __shfl_xor_sync(FULL, m2, o));
        gap = (float)(m1 - m2);
        if (gap > 1.0f) {
            for (int k = lane; k < K; k += 32)
                if (k != i1) S2 += expf((float)(s_xw[k] - m2));
            S2 = warp_sum(S2);
        }
    }
    double c_acc = 0.0;
    const double km1 = (double)(K - 1);
    for (int k = lane; k < K; k += 32) {
        const double xv = s_xw[k];
        const float e = expf((float)(xv - m1));
        const float wt = e * invS;
        c_acc -= (double)wt * xv;
        float gq = wt;
        if (EST == ZS_EST_VIMCO) {
            const float lq = s_lq[k];
            const float mu_m = (float)((sumd - (xv - m1)) / km1);
            float sig;
            if (k == i1 && gap > 1.0f) {
                // the arg-max row: S - e would cancel, re-centre on the second max (mu_m is relative to m1)
                const float Sloo = S2 + expf(mu_m + gap);
                sig = gap + (logf(S) - logf(Sloo));
            } else {
                sig = -log1pf((expf(mu_m) - e) * invS);
            }
            c_acc -= (double)lq * (double)sig;
            gq = wt - sig;
        }
        if (dlogp) dlogp[(int64_t)k * B + b] = -wt * gscale;
        if (dlogq) dlogq[(int64_t)k * B + b] = gq * gscale;
        if (logpx_out) logpx_out[(int64_t)k * B + b] = s_lpx[k];
    }
    c_acc = warp_sum(c_acc);
    // accumulate: running sum of the column's objective over launches (one writer per column: deterministic)
    const float cval = (float)c_acc * cscale;  // every lane holds the column's total
    if (lane == 0 && cost) cost[b] = prev_cost + cval;
    return cval;
}

// The mean objective itself (sum_b cost_b) without another launch.  Every objective warp keeps the double sum of the
// (float-rounded) column costs it wrote -- its columns and their order are fixed by the grid -- and, when its last
// column is done, stores that partial sum into its slot of the caller's workspace and takes a ticket.  The warp that
// draws the last of the 2 x gridDim.x tickets adds the 2 x gridDim.x partial sums in slot order (lane-strided, shuffle
// tree: the result does not depend on which warp does it), stores the float and re-arms the counter for the next launch
// on this stream.  One batch of <= 10 loads per lane, issued while the row warps still write the last column's
// gradient.  Workspace (ZS_FUSED_LOSS_WS_BYTES, zero-initialised once, one per stream): word 0 = ticket, then from
// byte 8 the double partial sums.
__device__ __forceinline__ void finish_loss(int lane, int p, double part, float* __restrict__ loss_out,
                                            unsigned* __restrict__ ws) {
    if (loss_out == nullptr) return;
    double* partial = reinterpret_cast<double*>(ws + 2);
    unsigned t = 0;
    if (lane == 0) {
        __stcg(partial + 2 * blockIdx.x + p, part);
        __threadfence();
        t = atomicAdd(ws, 1u);
    }
    t = __shfl_sync(0xffffffffu, t, 0);
    const unsigned n = 2u * gridDim.x;
    if (t != n - 1u) return;
    __threadfence();
    double v[ZS_FUSED_LOSS_MAX_GRID * 2 / 32];
#pragma unroll
    for (int i = 0; i < ZS_FUSED_LOSS_MAX_GRID * 2 / 32; ++i) {
        const unsigned idx = (unsigned)lane + 32u * i;
        v[i] = idx < n ? __ldcg(partial + idx) : 0.0;
    }
    double acc = 0.0;
#pragma unroll
    for (int i = 0; i < ZS_FUSED_LOSS_MAX_GRID * 2 / 32; ++i) acc += v[i];
    acc = warp_sum(acc);
    if (lane == 0) {
        *loss_out = (float)acc;
        *ws = 0u;
    }
}

// ---------------------------------------------------------------------------------------------
// Ring variant (fallback for shapes the box kernels do not take): one persistent CTA per SM, warp-specialised.
//   row warps      : warp w owns rows k = w, w+NW, ... of every column and a private mini-ring of D
//                    shared-memory row slots.  Its task stream is
//                       A(c,k)  first read of the row   (HBM)  -> log-pmf
//                       B(c,k)  second read of the row  (L2 hit: only ~2 columns per SM are in flight,
//                                                        ~46 MB chip-wide)  -> dprobs
//                    Rows arrive by 1-D bulk async copies (cp.async.bulk + mbarrier complete_tx) that the
//                    warp issues itself, D tasks ahead, each time it has consumed a slot: the bytes in
//                    flight live in shared memory (NW*D*X*4, ~150 KB), not in registers, and A(c+1) loads
//                    overlap B(c) stores.  Each row warp derives max / sum-exp of the column redundantly,
//                    so the only CTA-wide rendezvous per column is one named barrier after phase A.
//   stager warp    : stages the observation row x and the per-column scalars of the columns ahead.
//   objective warps: two, alternating columns: cost, dlogp, dlogq of a column, with two column periods
//                    to finish — off the row warps' critical path.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Named barrier over a subset of the CTA's warps (nthreads = 32 * participating warps).  The warp is
// re-converged first and the non-.aligned form is used, so a lane-0-only branch just before the
// rendezvous (issue_next) cannot make the arrival divergent.
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    __syncwarp();
    asm volatile("barrier.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---- stager helpers: batched global loads ---------------------------------------------------------------
__device__ __forceinline__ void stage_scalars_batched(float* s_other, float* s_lq, const float* __restrict__ logp_other,
                                                      const float* __restrict__ logq, int K, int64_t B, int64_t b, int lane) {
    for (int k0 = lane; k0 < K; k0 += 32 * 4) {
        float o[4], q[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + 32 * u;
            const int kc = k < K ? k : k0;  // always in bounds
            o[u] = logp_other ? __ldg(logp_other + (int64_t)kc * B + b) : 0.f;
            q[u] = logq ? __ldg(logq + (int64_t)kc * B + b) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int k = k0 + 32 * u;
            if (k < K) {
                s_other[k] = o[u];
                s_lq[k] = q[u];
            }
        }
    }
}
// An x slot holds two arrays of X floats.  Binary x (every element 0 or 1): c = 1 - x and e = (x == 1 ? +1e-8 : -1e-8);
// the signed log argument t = (p - c) + e then equals p + eps (x = 1) or -((1 - p) + eps) (x = 0) bit for bit, so
// the row loops need two adds per element instead of compare / subtract / select / add.  Other x: the row itself
// in the first array.  The flag must be known before anything is written: rows of up to 1024 floats are held in
// registers meanwhile, longer rows are read twice (the second read is an L1/L2 hit).
__device__ __forceinline__ void stage_x_write(float4* dst, float4* dst_e, int v, const float4& t, bool binary) {
    if (binary) {
        dst[v] = make_float4(1.0f - t.x, 1.0f - t.y, 1.0f - t.z, 1.0f - t.w);
        dst_e[v] = make_float4(t.x == 1.f ? 1e-8f : -1e-8f, t.y == 1.f ? 1e-8f : -1e-8f, t.z == 1.f ? 1e-8f : -1e-8f,
                               t.w == 1.f ? 1e-8f : -1e-8f);
    } else {
        dst[v] = t;
    }
}
__device__ __forceinline__ bool stage_x_is_binary(const float4& t) {
    return (t.x == 0.f || t.x == 1.f) && (t.y == 0.f || t.y == 1.f) && (t.z == 0.f || t.z == 1.f) && (t.w == 0.f || t.w == 1.f);
}
__device__ __forceinline__ void stage_x_batched(float* s_xrow, int* s_flag, const float* __restrict__ xrow, int X4, int lane) {
    const float4* src = reinterpret_cast<const float4*>(xrow);
    float4* dst = reinterpret_cast<float4*>(s_xrow);
    float4* dst_e = dst + X4;
    bool binary = true;
    if (X4 <= 32 * 8) {
        float4 t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int v = lane + 32 * u;
            t[u] = __ldg(src + (v < X4 ? v : 0));  // always in bounds
            binary = binary && stage_x_is_binary(t[u]);
        }
        binary = __all_sync(0xffffffffu, binary);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int v = lane + 32 * u;
            if (v < X4) stage_x_write(dst, dst_e, v, t[u], binary);
        }
    } else {
        for (int v0 = lane; v0 < X4; v0 += 32 * 8) {
            float4 t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int v = v0 + 32 * u;
                t[u] = __ldg(src + (v < X4 ? v : v0));
                binary = binary && stage_x_is_binary(t[u]);
            }
        }
        binary = __all_sync(0xffffffffu, binary);
        for (int v0 = lane; v0 < X4; v0 += 32 * 8) {
            float4 t[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int v = v0 + 32 * u;
                t[u] = __ldg(src + (v < X4 ? v : v0));
            }
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int v = v0 + 32 * u;
                if (v < X4) stage_x_write(dst, dst_e, v, t[u], binary);
            }
        }
    }
    if (lane == 0) *s_flag = binary ? 1 : 0;
}

// All CTAs of these persistent kernels otherwise run their read-heavy and write-heavy phases in lock-step
// (measured with %globaltimer: every SM is in the same phase for the first three columns), which leaves HBM
// reads idle in one phase and over-subscribed in the other.  CTA i starts (i mod groups) * cycles late.
__device__ __forceinline__ void stagger_start(int groups, int cycles) {
    if (groups > 1) {
        const long long wait = (long long)(blockIdx.x % groups) * cycles;
        const long long t0 = clock64();
        while (clock64() - t0 < wait) {}
    }
}

struct RingLayout {
    int K, X, R, Kpad;
    __host__ __device__ RingLayout(int K_, int X_, int R_) : K(K_), X(X_), R(R_), Kpad((K_ + 3) & ~3) {}
    __host__ __device__ size_t slots_off() const { return 0; }
    __host__ __device__ size_t x_off() const { return (size_t)R * X * 4; }
    __host__ __device__ size_t xw_off() const { return (x_off() + (size_t)6 * X * 4 + 15) & ~(size_t)15; }
    __host__ __device__ size_t xv_off() const { return xw_off() + (size_t)2 * Kpad * 8; }     // xw: [2][Kpad] double
    __host__ __device__ size_t lpx_off() const { return xv_off() + (size_t)4 * Kpad * 8; }    // xv: [4][Kpad] double
    __host__ __device__ size_t other_off() const { return lpx_off() + (size_t)4 * Kpad * 4; }  // [4][Kpad]
    __host__ __device__ size_t lq_off() const { return other_off() + (size_t)4 * Kpad * 4; }
    __host__ __device__ size_t bin_off() const { return lq_off() + (size_t)4 * Kpad * 4; }
    __host__ __device__ size_t bar_off() const { return (bin_off() + 16 + 15) & ~(size_t)15; }
    __host__ __device__ size_t total() const { return bar_off() + (size_t)R * 8; }
};

// ---- row loops of the ring kernel ---------------------------------------------------------------------
// The kernel is issue/latency-bound on an SM well before HBM saturates (37 CTAs alone run at the same
// 8.5 us per column as 148 do: profiles/r1_notes.md), so these loops are written for instruction count:
//  * binary x: log2 of the PRODUCT of four selected arguments (one SFU op per 4 elements; arguments are
//    >= 1e-8 for valid probabilities, so the product cannot underflow); the reference's "a log argument is
//    negative -> NaN" rule is kept exactly by tracking min / max of p (valid iff -1e-8 <= p <= 1) with two
//    3-input min/max per 4 elements instead of forming both arguments;
//  * backward: d/dp = g / s with the signed argument s = x ? p + eps : (p - 1) - eps == -((1 - p) + eps);
//  * ITER > 0 is the exact compile-time trip count ceil(X/128) per lane: fully unrolled, constant offsets,
//    no remainder loop (the remainder loops were a quarter of all instructions executed).
// x4 points at an x slot (see stage_x_batched).  The ring reads shared memory twice per row and is bound by
// that (measured: the two-array form costs 8 us per launch here), so its binary path reads c only and selects.
template <bool BINARY>
__device__ __forceinline__ void ring_lpmf4(const float4* x4, int X4, int v, const float4& p, float& acc, float& pmin,
                                           float& pmax) {
    if (BINARY) {
        const float4 c = lds128(x4 + v);  // c = 1 - x
        const float a0 = (c.x == 0.f ? p.x : 1.0f - p.x) + 1e-8f, a1 = (c.y == 0.f ? p.y : 1.0f - p.y) + 1e-8f;
        const float a2 = (c.z == 0.f ? p.z : 1.0f - p.z) + 1e-8f, a3 = (c.w == 0.f ? p.w : 1.0f - p.w) + 1e-8f;
        acc += fast_log2((a0 * a1) * (a2 * a3));
        pmin = fminf(pmin, fminf(p.x, p.y));
        pmin = fminf(pmin, fminf(p.z, p.w));
        pmax = fmaxf(pmax, fmaxf(p.x, p.y));
        pmax = fmaxf(pmax, fmaxf(p.z, p.w));
    } else {
        float mn = 1.0f;
        acc += lpmf4<false>(p, lds128(x4 + v), mn);
    }
}
template <bool BINARY>
__device__ __forceinline__ float4 ring_dprobs4(const float4* x4, int X4, int v, const float4& p, float g) {
    if (BINARY) {
        const float4 c = lds128(x4 + v);
        float4 o;
        o.x = g * fast_rcp(c.x == 0.f ? p.x + 1e-8f : (p.x - 1.0f) - 1e-8f);
        o.y = g * fast_rcp(c.y == 0.f ? p.y + 1e-8f : (p.y - 1.0f) - 1e-8f);
        o.z = g * fast_rcp(c.z == 0.f ? p.z + 1e-8f : (p.z - 1.0f) - 1e-8f);
        o.w = g * fast_rcp(c.w == 0.f ? p.w + 1e-8f : (p.w - 1.0f) - 1e-8f);
        return o;
    }
    return dprobs4<false>(p, lds128(x4 + v), g);
}

template <bool BINARY, int ITER>
__device__ __forceinline__ float smem_row_logpmf(const float4* __restrict__ p4, const float4* __restrict__ x4, int X4,
                                                 int lane) {
    float acc = 0.f, pmin = 0.f, pmax = 0.f;  // 0 is inside the valid range of p
    if (ITER > 0) {
#pragma unroll
        for (int u = 0; u < ITER; ++u) {
            const int v = lane + 32 * u;
            if (u + 1 < ITER || v < X4) ring_lpmf4<BINARY>(x4, X4, v, lds128(p4 + v), acc, pmin, pmax);
        }
    } else {
#pragma unroll 4
        for (int v = lane; v < X4; v += 32) ring_lpmf4<BINARY>(x4, X4, v, lds128(p4 + v), acc, pmin, pmax);
    }
    // a negative log argument is NaN in the reference: p + eps < 0 or (1 - p) + eps < 0
    if (BINARY && (pmin < -1e-8f || pmax > 1.0f)) acc = __int_as_float(0x7fc00000);
    return acc;
}
template <bool BINARY, int ITER>
__device__ __forceinline__ void smem_row_dprobs(float* __restrict__ drow, const float4* __restrict__ p4,
                                                const float4* __restrict__ x4, int X4, int lane, float g) {
    if (ITER > 0) {
#pragma unroll
        for (int u = 0; u < ITER; ++u) {
            const int v = lane + 32 * u;
            if (u + 1 < ITER || v < X4) stg_hint(drow + 4 * v, ring_dprobs4<BINARY>(x4, X4, v, lds128(p4 + v), g), 0);
        }
    } else {
#pragma unroll 4
        for (int v = lane; v < X4; v += 32) stg_hint(drow + 4 * v, ring_dprobs4<BINARY>(x4, X4, v, lds128(p4 + v), g), 0);
    }
}

// max and 1/sum-exp of a column's posted log-weights (every row warp, redundantly)
__device__ __forceinline__ void ring_max_sumexp(int lane, int K, const double* s_xv, double& m1, float& invS) {
    float mf = -INFINITY;
    for (int k = lane; k < K; k += 32) mf = fmaxf(mf, (float)s_xv[k]);
    mf = warp_max(mf);
    m1 = (double)mf;
    float S = 0.f;
    for (int k = lane; k < K; k += 32) S += expf((float)(s_xv[k] - m1));
    S = warp_sum(S);
    invS = fast_rcp(S) * (2.0f - S * fast_rcp(S));
}

#ifndef ZS_RING_EARLY_DEFAULT
#define ZS_RING_EARLY_DEFAULT 0
#endif
#ifndef ZS_RING_MAX_ROW_WARPS
#define ZS_RING_MAX_ROW_WARPS 25  // + 3 service warps = 896 threads: 72 registers per thread
#endif
// (A variant that read the second pass with plain L2 loads instead of a second bulk copy was measured at
// 77-88 us against 67-74 us: the exposed L2 latency costs more than the copy engine saves; removed.)
template <int EST, int ITER>
__global__ void __launch_bounds__((ZS_RING_MAX_ROW_WARPS + 3) * 32, 1)
    k_iw_bernoulli_ring(float* __restrict__ cost, float* __restrict__ dprobs, float* __restrict__ dlogp,
                        float* __restrict__ dlogq, float* __restrict__ logpx_out, const float* __restrict__ probs,
                        const float* __restrict__ x, const float* __restrict__ logp_other,
                        const float* __restrict__ logq, int K, int64_t B, int X, int R, float gscale,
                        int stagger_groups, int stagger_cycles, int flags, long long* __restrict__ trace, int64_t ldkb,
                        float* __restrict__ loss_out, unsigned* __restrict__ ticket) {
    extern __shared__ __align__(128) unsigned char smem[];
    stagger_start(stagger_groups, stagger_cycles);
    const RingLayout L(K, X, R);
    const int Kpad = L.Kpad;
    float* slots = reinterpret_cast<float*>(smem + L.slots_off());
    float* s_x = reinterpret_cast<float*>(smem + L.x_off());
    double* s_xw = reinterpret_cast<double*>(smem + L.xw_off());
    double* s_xv = reinterpret_cast<double*>(smem + L.xv_off());  // log-weights of a column, posted by the row warps
    float* s_lpx = reinterpret_cast<float*>(smem + L.lpx_off());
    float* s_other = reinterpret_cast<float*>(smem + L.other_off());
    float* s_lq = reinterpret_cast<float*>(smem + L.lq_off());
    int* s_bin = reinterpret_cast<int*>(smem + L.bin_off());
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bar_off());

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // warp roles: [0, NW) row warps | NW stager | NW+1, NW+2 objective warps for even / odd columns
    const int NW = (blockDim.x >> 5) - 3;
    const bool is_stager = warp == NW, is_obj = warp > NW;
    const int X4 = X >> 2;
    const uint32_t row_bytes = (uint32_t)X * 4u;
    const float LN2 = 0.6931471805599453f;
    const int phases = dprobs ? 2 : 1;  // row tasks per column that travel through the ring
    const int64_t ncols = ((int64_t)blockIdx.x < B) ? (B - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    auto mark = [&](int col, int point) {
        if (trace != nullptr && threadIdx.x == 0 && col < 8)
            trace[(int64_t)blockIdx.x * 40 + col * 5 + point] = clock64();
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < R; ++s) mbar_init(&full[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // ---- row-warp prefetch cursor.  Warp w owns the D slots [w*D, w*D+D) and its row tasks, in order
    //   A(c, w), A(c, w+NW), ..., B(c, w), B(c, w+NW), ..., A(c+1, w), ...
    // (A = first read, HBM; B = second read of the same row, an L2 hit;).
    // The first D copies are issued BEFORE the stager's first (dependent, cold) global loads so the
    // HBM pipe fills while x and the [K] scalars are staged.
    const int D = R / NW;
    const int my_rows = warp < NW ? (K - warp + NW - 1) / NW : 0;
    int64_t pf_c = 0, pf_b = blockIdx.x;
    int pf_ph = 0, pf_j = 0, pf_pos = 0;
    auto issue_next = [&]() {
        if (pf_c >= ncols || my_rows == 0) return;
        const int k = warp + pf_j * NW;
        const int s = warp * D + pf_pos;
        mbar_expect_tx(&full[s], row_bytes);
        bulk_load(slots + (size_t)s * X, probs + ((int64_t)k * B + pf_b) * X, row_bytes, &full[s]);
        if (++pf_pos == D) pf_pos = 0;
        if (++pf_j == my_rows) {
            pf_j = 0;
            if (++pf_ph == phases) { pf_ph = 0; ++pf_c; pf_b += gridDim.x; }
        }
    };
    const bool early_issue = (flags & FUSED_EARLY_ISSUE) != 0;  // dev knob
    if (early_issue && warp < NW && lane == 0)
        for (int i = 0; i < D; ++i) issue_next();
    // Per-column scalars and log-pmf live in 4 buffers (column & 3), the x row in 3 (column % 3):
    // an objective warp may work on column c until the barrier of column c+2.
    // The stager takes part in every column rendezvous, so one iteration of its loop bounds the column rate:
    // its global loads are issued in batches (all in flight together), never one latency after the other.
    auto stage_scalars = [&](int64_t b, int buf) { stage_scalars_batched(s_other + buf * Kpad, s_lq + buf * Kpad, logp_other, logq, K, ldkb, b, lane); };
    auto stage_x = [&](int64_t b, int slot) { stage_x_batched(s_x + (size_t)slot * 2 * X, s_bin + slot, x + b * X, X4, lane); };
    if (is_stager && ncols > 0) {
        stage_scalars(blockIdx.x, 0);
        stage_x(blockIdx.x, 0);
        if (ncols > 1) {
            stage_scalars((int64_t)blockIdx.x + gridDim.x, 1);
            stage_x((int64_t)blockIdx.x + gridDim.x, 1);
        }
    }
    __syncthreads();
    if (!early_issue && warp < NW && lane == 0)
        for (int i = 0; i < D; ++i) issue_next();

    // column c rendezvous on named barrier 1 + (c & 1): row warps, the stager and the objective warp
    // of that parity
    const int sync_threads = (NW + 2) * 32;
    if (is_stager) {
        int64_t b = blockIdx.x;
        for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
            named_bar_sync(1 + (int)(c & 1), sync_threads);
            // a row warp posts the log-weight of a row of column c+1 as soon as it is reduced, so the
            // scalars are staged two columns ahead (into the buffer of column c-2, dead by now)
            if (c + 2 < ncols) {
                stage_scalars(b + 2 * (int64_t)gridDim.x, (int)((c + 2) & 3));
                stage_x(b + 2 * (int64_t)gridDim.x, (int)((c + 2) % 3));
            }
        }
        return;
    }
    if (is_obj) {
        // ---- objective warps: cost / dlogp / dlogq of every other column ----------------------------
        const int p = warp - NW - 1;
        int64_t b = (int64_t)blockIdx.x + (int64_t)p * gridDim.x;
        double part = 0.0;
        for (int64_t c = p; c < ncols; c += 2, b += 2 * (int64_t)gridDim.x) {
            const int buf = (int)(c & 3);
            named_bar_sync(1 + p, sync_threads);  // lpx of column c complete
            part += (double)column_objective<EST>(lane, K, ldkb, b, s_lpx + buf * Kpad, s_other + buf * Kpad,
                                                  s_lq + buf * Kpad, s_xw + p * Kpad, gscale, cost, dlogp, dlogq,
                                                  logpx_out, flags);
        }
        finish_loss(lane, p, part, loss_out, ticket);
        return;
    }

    // ---- row warps.  After consuming a slot the warp itself re-arms the slot's mbarrier and issues the
    // bulk copy of the task D ahead, so up to D rows per warp are in flight in shared memory and the loads
    // of the next column overlap the stores of this one.  A slot is filled and waited on by one warp only,
    // so its mbarrier phases are always observed in sequence.
    int ring_pos = 0;         // consumer cursor in the warp's mini-ring
    uint32_t ring_phase = 0;  // parity of the fill being waited for
    int64_t b = blockIdx.x;
    for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
        const int par = (int)(c & 3), xs = (int)(c % 3);
        const float4* x4 = reinterpret_cast<const float4*>(s_x + (size_t)xs * 2 * X);
        const bool binary = s_bin[xs] != 0;
        mark((int)c, 0);
        // ---- phase A: log-pmf of the owned rows as they land ---------------------------------------
        for (int k = warp; k < K; k += NW) {
            const int s = warp * D + ring_pos;
            mbar_wait(&full[s], ring_phase);
            if (++ring_pos == D) { ring_pos = 0; ring_phase ^= 1u; }
            const float4* p4 = reinterpret_cast<const float4*>(slots + (size_t)s * X);
            float acc = binary ? smem_row_logpmf<true, ITER>(p4, x4, X4, lane) : smem_row_logpmf<false, ITER>(p4, x4, X4, lane);
            acc = warp_sum(acc);  // every lane has finished reading the slot
            if (lane == 0) {
                issue_next();
                const float lp = acc * LN2;
                s_lpx[par * Kpad + k] = lp;
                // same association as k_iw_objective: (logp - logq) + extra, in double
                s_xv[par * Kpad + k] = ((double)lp - (double)s_lq[par * Kpad + k]) + (double)s_other[par * Kpad + k];
            }
        }
        mark((int)c, 1);
        named_bar_sync(1 + (int)(c & 1), sync_threads);
        mark((int)c, 2);
        if (dprobs) {
            // ---- phase B: weights of the owned rows, rows again (L2) -> dprobs ----------------------
            double m1;
            float invS;
            ring_max_sumexp(lane, K, s_xv + par * Kpad, m1, invS);
            for (int k = warp; k < K; k += NW) {
                const float g = -(expf((float)(s_xv[par * Kpad + k] - m1)) * invS) * gscale;
                float* drow = dprobs + ((int64_t)k * B + b) * X;
                const int s = warp * D + ring_pos;
                mbar_wait(&full[s], ring_phase);
                if (++ring_pos == D) { ring_pos = 0; ring_phase ^= 1u; }
                const float4* p4 = reinterpret_cast<const float4*>(slots + (size_t)s * X);
                if (binary) smem_row_dprobs<true, ITER>(drow, p4, x4, X4, lane, g);
                else smem_row_dprobs<false, ITER>(drow, p4, x4, X4, lane, g);
                __syncwarp();
                if (lane == 0) issue_next();
            }
        }
        mark((int)c, 3);
    }
}

// ---------------------------------------------------------------------------------------------
// Generic box variant (run-time geometry; the fixed-geometry kernel further down is the default): the column is
// RESIDENT in shared memory between its two passes and arrives by TENSOR bulk copies.
//
// Why (tools/probes/tma_probe.cu, tma_tensor_probe.cu, profiles/r1_notes.md): every variant of the ring
// kernel ran at 8.5 us per column per SM, with 37 CTAs as with 148, with or without the arithmetic.  The
// bound was the SM's copy engine: a 1-D cp.async.bulk costs ~134 cycles of fixed overhead, so 3 KB row copies
// peak at 38 GB/s per SM, below the 43 GB/s per SM that HBM can feed, and the ring issued 100 of them per
// column.  A 3-D tensor copy moves a box {inner, 1, K} -- the same `inner` floats of all K rows of one batch
// column -- with one instruction at ~13 cycles per row segment: 64 GB/s per SM at 448-byte segments, 105 GB/s
// at 784.  The column is cut into X/inner boxes that flow through a ring of NSLOT > X/inner slots:
//   phase A(c)  waits for the boxes of column c in order, adds up the log-pmf pieces of the warp's two rows;
//   rendezvous  (named barrier, as in the ring kernel; objective + stager warps unchanged);
//   phase B(c)  walks the still-resident boxes again, writes dprobs, releases each box (empty mbarrier);
//   producer    one thread refills a released slot with the box NSLOT tasks ahead: every box is requested
//               about (NSLOT+1)/(2 NBOX) of a column period before its first read.
// probs is read from L2/HBM exactly once; no second pass over L2.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_load_box(void* dst_smem, const CUtensorMap* map, int c0, int c1, int c2,
                                             uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(
            smem_u32(dst_smem)),
        "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar))
        : "memory");
}

// tma_load_box with an L2 cache policy (createpolicy), e.g. evict-first for data that is read exactly once
__device__ __forceinline__ void tma_load_box_hint(void* dst_smem, const CUtensorMap* map, int c0, int c1, int c2,
                                                  uint64_t* bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3, %4}], [%5], %6;" ::"r"(
            smem_u32(dst_smem)),
        "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}

// request a box into L2 only (no shared-memory destination, no completion tracking)
__device__ __forceinline__ void tma_prefetch_box_l2(const CUtensorMap* map, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2)
                 : "memory");
}

struct BoxLayout {
    int K, X, inner, nslot, Kpad;
    __host__ __device__ BoxLayout(int K_, int X_, int inner_, int nslot_)
        : K(K_), X(X_), inner(inner_), nslot(nslot_), Kpad((K_ + 3) & ~3) {}
    __host__ __device__ size_t slot_bytes() const { return ((size_t)K * inner * 4 + 127) & ~(size_t)127; }
    __host__ __device__ size_t slots_off() const { return 0; }
    __host__ __device__ size_t x_off() const { return (size_t)nslot * slot_bytes(); }
    __host__ __device__ size_t xw_off() const { return (x_off() + (size_t)6 * X * 4 + 15) & ~(size_t)15; }
    __host__ __device__ size_t xv_off() const { return xw_off() + (size_t)2 * Kpad * 8; }
    __host__ __device__ size_t lpx_off() const { return xv_off() + (size_t)4 * Kpad * 8; }
    __host__ __device__ size_t other_off() const { return lpx_off() + (size_t)4 * Kpad * 4; }
    __host__ __device__ size_t lq_off() const { return other_off() + (size_t)4 * Kpad * 4; }
    __host__ __device__ size_t bin_off() const { return lq_off() + (size_t)4 * Kpad * 4; }
    __host__ __device__ size_t bar_off() const { return (bin_off() + 16 + 15) & ~(size_t)15; }
    __host__ __device__ size_t total() const { return bar_off() + (size_t)2 * nslot * 8; }
};

// two rows of one box against the same x piece: one load of the c / e pieces serves both rows
template <bool BINARY>
__device__ __forceinline__ void box_lpmf_pair(const float4* xq, int X4, int v, const float4& pa, const float4& pb,
                                              float& acc_a, float& acc_b, float (&rng)[4]) {
    if (BINARY) {
        const float4 c = lds128(xq + v), e = lds128(xq + X4 + v);
        {
            const float t0 = (pa.x - c.x) + e.x, t1 = (pa.y - c.y) + e.y, t2 = (pa.z - c.z) + e.z, t3 = (pa.w - c.w) + e.w;
            acc_a += fast_log2(fabsf((t0 * t1) * (t2 * t3)));
            rng[0] = fminf(rng[0], fminf(pa.x, pa.y));
            rng[0] = fminf(rng[0], fminf(pa.z, pa.w));
            rng[1] = fmaxf(rng[1], fmaxf(pa.x, pa.y));
            rng[1] = fmaxf(rng[1], fmaxf(pa.z, pa.w));
        }
        {
            const float t0 = (pb.x - c.x) + e.x, t1 = (pb.y - c.y) + e.y, t2 = (pb.z - c.z) + e.z, t3 = (pb.w - c.w) + e.w;
            acc_b += fast_log2(fabsf((t0 * t1) * (t2 * t3)));
            rng[2] = fminf(rng[2], fminf(pb.x, pb.y));
            rng[2] = fminf(rng[2], fminf(pb.z, pb.w));
            rng[3] = fmaxf(rng[3], fmaxf(pb.x, pb.y));
            rng[3] = fmaxf(rng[3], fmaxf(pb.z, pb.w));
        }
    } else {
        const float4 xx = lds128(xq + v);
        float mn = 1.0f;
        acc_a += lpmf4<false>(pa, xx, mn);
        acc_b += lpmf4<false>(pb, xx, mn);
    }
}
template <bool BINARY>
__device__ __forceinline__ void box_dprobs_pair(const float4* xq, int X4, int v, const float4& pa, const float4& pb,
                                                float ga, float gb, float4& oa, float4& ob) {
    if (BINARY) {
        const float4 c = lds128(xq + v), e = lds128(xq + X4 + v);
        oa.x = ga * fast_rcp((pa.x - c.x) + e.x);
        oa.y = ga * fast_rcp((pa.y - c.y) + e.y);
        oa.z = ga * fast_rcp((pa.z - c.z) + e.z);
        oa.w = ga * fast_rcp((pa.w - c.w) + e.w);
        ob.x = gb * fast_rcp((pb.x - c.x) + e.x);
        ob.y = gb * fast_rcp((pb.y - c.y) + e.y);
        ob.z = gb * fast_rcp((pb.z - c.z) + e.z);
        ob.w = gb * fast_rcp((pb.w - c.w) + e.w);
    } else {
        const float4 xx = lds128(xq + v);
        oa = dprobs4<false>(pa, xx, ga);
        ob = dprobs4<false>(pb, xx, gb);
    }
}

constexpr int BOX_MAX_ROW_WARPS = 25;  // + stager, two objective warps, producer = 29 warps: 70 registers per thread

template <int EST>
__global__ void __launch_bounds__((BOX_MAX_ROW_WARPS + 4) * 32, 1)
    k_iw_bernoulli_box(const __grid_constant__ CUtensorMap probs_map, float* __restrict__ cost,
                       float* __restrict__ dprobs, float* __restrict__ dlogp, float* __restrict__ dlogq,
                       float* __restrict__ logpx_out, const float* __restrict__ x,
                       const float* __restrict__ logp_other, const float* __restrict__ logq, int K, int64_t B, int X,
                       int inner, int nslot, int l2_ahead, float gscale, int stagger_groups, int stagger_cycles,
                       int flags, long long* __restrict__ trace, int64_t ldkb, float* __restrict__ loss_out,
                       unsigned* __restrict__ ticket) {
    extern __shared__ __align__(128) unsigned char smem[];
    const BoxLayout L(K, X, inner, nslot);
    const int Kpad = L.Kpad;
    const uint32_t slot_bytes = (uint32_t)L.slot_bytes();
    unsigned char* slots = smem + L.slots_off();
    float* s_x = reinterpret_cast<float*>(smem + L.x_off());
    double* s_xw = reinterpret_cast<double*>(smem + L.xw_off());
    double* s_xv = reinterpret_cast<double*>(smem + L.xv_off());
    float* s_lpx = reinterpret_cast<float*>(smem + L.lpx_off());
    float* s_other = reinterpret_cast<float*>(smem + L.other_off());
    float* s_lq = reinterpret_cast<float*>(smem + L.lq_off());
    int* s_bin = reinterpret_cast<int*>(smem + L.bin_off());
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bar_off());
    uint64_t* empty = full + nslot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // warp roles: [0, NW) row warps | NW stager | NW+1, NW+2 objective warps (even / odd columns) | NW+3 producer
    const int NW = (blockDim.x >> 5) - 4;
    const int X4 = X >> 2, inner4 = inner >> 2, nbox = X / inner;
    const uint32_t box_bytes = (uint32_t)K * (uint32_t)inner * 4u;
    const float LN2 = 0.6931471805599453f;
    const int64_t ncols = ((int64_t)blockIdx.x < B) ? (B - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
    auto mark = [&](int col, int point) {
        if (trace != nullptr && threadIdx.x == 0 && col < 8)
            trace[(int64_t)blockIdx.x * 40 + col * 5 + point] = clock64();
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < nslot; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], (uint32_t)NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // The stager takes part in every column rendezvous, so one iteration of its loop bounds the column rate:
    // its global loads are issued in batches (all in flight together), never one latency after the other.
    auto stage_scalars = [&](int64_t b, int buf) { stage_scalars_batched(s_other + buf * Kpad, s_lq + buf * Kpad, logp_other, logq, K, ldkb, b, lane); };
    auto stage_x = [&](int64_t b, int slot) { stage_x_batched(s_x + (size_t)slot * 2 * X, s_bin + slot, x + b * X, X4, lane); };
    const bool is_stager = warp == NW, is_obj = warp == NW + 1 || warp == NW + 2, is_producer = warp == NW + 3;
    stagger_start(stagger_groups, stagger_cycles);
    if (is_stager && ncols > 0) {
        stage_scalars(blockIdx.x, 0);
        stage_x(blockIdx.x, 0);
        if (ncols > 1) {
            stage_scalars((int64_t)blockIdx.x + gridDim.x, 1);
            stage_x((int64_t)blockIdx.x + gridDim.x, 1);
        }
    }
    __syncthreads();

    if (is_producer) {
        // ---- producer: box t = (column t / nbox, piece t % nbox) goes to slot t % nslot.  Slots free up only
        // while phase B runs, so before it blocks the producer asks L2 for the boxes of the next `l2_ahead`
        // tasks: HBM then streams the next column during phase A as well, and the later copies are L2 hits.
        if (lane == 0) {
            int slot = 0, q = 0, pq = 0;
            uint32_t wait_parity = 1;  // first pass over the ring: nothing to wait for
            bool first_pass = true;
            int64_t col = blockIdx.x, pcol = blockIdx.x;
            const int64_t ntask = ncols * nbox;
            int64_t pt = 0;  // next task to prefetch into L2
            for (int64_t t = 0; t < ntask; ++t) {
                if (l2_ahead > 0 && !first_pass) {
                    if (pt < t) {  // never behind the real copies
                        const int64_t skip = t - pt;
                        pt = t;
                        pq = q;
                        pcol = col;
                        (void)skip;
                    }
                    for (; pt < ntask && pt < t + l2_ahead; ++pt) {
                        tma_prefetch_box_l2(&probs_map, pq * inner, (int)pcol, 0);
                        if (++pq == nbox) { pq = 0; pcol += gridDim.x; }
                    }
                }
                if (!first_pass) mbar_wait(&empty[slot], wait_parity);
                mbar_expect_tx(&full[slot], box_bytes);
                tma_load_box(slots + (size_t)slot * slot_bytes, &probs_map, q * inner, (int)col, 0, &full[slot]);
                if (++q == nbox) { q = 0; col += gridDim.x; }
                if (++slot == nslot) {
                    slot = 0;
                    if (first_pass) { first_pass = false; wait_parity = 0; }
                    else wait_parity ^= 1u;
                }
            }
        }
        return;
    }
    // column c rendezvous on named barrier 1 + (c & 1): row warps, the stager and the objective warp of that parity
    const int sync_threads = (NW + 2) * 32;
    if (is_stager) {
        int64_t b = blockIdx.x;
        for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
            named_bar_sync(1 + (int)(c & 1), sync_threads);
            // log-weights of column c+1 are posted during its phase A: scalars are staged two columns ahead
            if (c + 2 < ncols) {
                stage_scalars(b + 2 * (int64_t)gridDim.x, (int)((c + 2) & 3));
                stage_x(b + 2 * (int64_t)gridDim.x, (int)((c + 2) % 3));
            }
        }
        return;
    }
    if (is_obj) {
        const int p = warp - NW - 1;
        int64_t b = (int64_t)blockIdx.x + (int64_t)p * gridDim.x;
        double part = 0.0;
        for (int64_t c = p; c < ncols; c += 2, b += 2 * (int64_t)gridDim.x) {
            const int buf = (int)(c & 3);
            named_bar_sync(1 + p, sync_threads);  // lpx of column c complete
            part += (double)column_objective<EST>(lane, K, ldkb, b, s_lpx + buf * Kpad, s_other + buf * Kpad,
                                                  s_lq + buf * Kpad, s_xw + p * Kpad, gscale, cost, dlogp, dlogq,
                                                  logpx_out, flags);
        }
        finish_loss(lane, p, part, loss_out, ticket);
        return;
    }

    // ---- row warps: rows ka = warp and kb = warp + NW of every column (kb may not exist) ----------------
    const int ka = warp, kb = warp + NW;
    const bool has_b = kb < K;
    const int kb_eff = has_b ? kb : ka;  // a warp without a second row recomputes row a and drops the result
    int slot = 0;          // slot of the next box to be read for the first time
    uint32_t fparity = 0;  // parity of that fill
    int64_t b = blockIdx.x;
    for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
        const int par = (int)(c & 3), xs = (int)(c % 3);
        const float4* x4 = reinterpret_cast<const float4*>(s_x + (size_t)xs * 2 * X);
        const bool binary = s_bin[xs] != 0;
        const int slot0 = slot;  // first box of this column
        mark((int)c, 0);
        // ---- phase A ---------------------------------------------------------------------------------
        float acc_a = 0.f, acc_b = 0.f;
        float rng[4] = {0.f, 0.f, 0.f, 0.f};  // min / max of p per row (0 is inside the valid range)
        for (int q = 0; q < nbox; ++q) {
            mbar_wait(&full[slot], fparity);
            const float4* base = reinterpret_cast<const float4*>(slots + (size_t)slot * slot_bytes);
            const float4* pa4 = base + (size_t)ka * inner4;
            const float4* pb4 = base + (size_t)kb_eff * inner4;
            const float4* xq = x4 + q * inner4;
            if (binary) {
                for (int v = lane; v < inner4; v += 32)
                    box_lpmf_pair<true>(xq, X4, v, lds128(pa4 + v), lds128(pb4 + v), acc_a, acc_b, rng);
            } else {
                for (int v = lane; v < inner4; v += 32)
                    box_lpmf_pair<false>(xq, X4, v, lds128(pa4 + v), lds128(pb4 + v), acc_a, acc_b, rng);
            }
            if (!dprobs) {  // forward only: the box is dead after its first read
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[slot]);
            }
            if (++slot == nslot) { slot = 0; fparity ^= 1u; }
        }
        if (binary) {
            // a negative log argument is NaN in the reference: p + eps < 0 or (1 - p) + eps < 0
            if (rng[0] < -1e-8f || rng[1] > 1.0f) acc_a = __int_as_float(0x7fc00000);
            if (rng[2] < -1e-8f || rng[3] > 1.0f) acc_b = __int_as_float(0x7fc00000);
        }
        acc_a = warp_sum(acc_a);
        acc_b = warp_sum(acc_b);
        if (lane == 0) {
            // log-pmf -> s_lpx; log-weight, same association as k_iw_objective, in double -> s_xv
            const float la = acc_a * LN2;
            s_lpx[par * Kpad + ka] = la;
            s_xv[par * Kpad + ka] = ((double)la - (double)s_lq[par * Kpad + ka]) + (double)s_other[par * Kpad + ka];
            if (has_b) {
                const float lb = acc_b * LN2;
                s_lpx[par * Kpad + kb] = lb;
                s_xv[par * Kpad + kb] = ((double)lb - (double)s_lq[par * Kpad + kb]) + (double)s_other[par * Kpad + kb];
            }
        }
        mark((int)c, 1);
        named_bar_sync(1 + (int)(c & 1), sync_threads);
        mark((int)c, 2);
        if (dprobs) {
            // ---- phase B: weights of the two rows, dprobs from the resident boxes, release them -------
            double m1;
            float invS;
            ring_max_sumexp(lane, K, s_xv + par * Kpad, m1, invS);
            const float ga = -(expf((float)(s_xv[par * Kpad + ka] - m1)) * invS) * gscale;
            const float gb = -(expf((float)(s_xv[par * Kpad + kb_eff] - m1)) * invS) * gscale;
            float* da = dprobs + ((int64_t)ka * B + b) * X;
            float* db = dprobs + ((int64_t)kb_eff * B + b) * X;
            int bs = slot0;
            for (int q = 0; q < nbox; ++q) {
                const float4* base = reinterpret_cast<const float4*>(slots + (size_t)bs * slot_bytes);
                const float4* pa4 = base + (size_t)ka * inner4;
                const float4* pb4 = base + (size_t)kb_eff * inner4;
                const float4* xq = x4 + q * inner4;
                for (int v = lane; v < inner4; v += 32) {
                    float4 oa, ob;
                    if (binary) box_dprobs_pair<true>(xq, X4, v, lds128(pa4 + v), lds128(pb4 + v), ga, gb, oa, ob);
                    else box_dprobs_pair<false>(xq, X4, v, lds128(pa4 + v), lds128(pb4 + v), ga, gb, oa, ob);
                    stg_hint(da + q * inner + 4 * v, oa, 0);
                    if (has_b) stg_hint(db + q * inner + 4 * v, ob, 0);
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[bs]);
                if (++bs == nslot) bs = 0;
            }
        }
        mark((int)c, 3);
    }
}

// ---------------------------------------------------------------------------------------------
// Fixed-geometry box kernel.  ncu on the generic box kernel (profiles/r2_box_kernel_ncu.md): 45.6 k warp
// instructions per column and SM at 65 % issue utilisation -- the kernel was ISSUE-bound, and 40 % of the
// row warps' instructions were address arithmetic and loop control around run-time box geometry.  Here the
// box width (INNER4 float4 per row piece) and the boxes per column (NBOX) are template parameters: the box
// loops are fully unrolled, every shared-memory access is a 32-bit base register plus an immediate, every
// global store a 64-bit row pointer plus an immediate.  Roles, barriers and numerics are those of
// k_iw_bernoulli_box; the prologue stages only column 0 before the first rendezvous.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float4 lds128_u32(uint32_t addr) {
    float4 r;
    asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "r"(addr));
    return r;
}
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "ZS_WAITU:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra ZS_DONEU;\n"
        "bra ZS_WAITU;\n"
        "ZS_DONEU:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

__device__ __forceinline__ void sts128_u32(uint32_t addr, const float4& v) {
    asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ float4 sigmoid4(const float4& l) {
    return make_float4(fast_sigmoid(l.x), fast_sigmoid(l.y), fast_sigmoid(l.z), fast_sigmoid(l.w));
}
// p (1 - p), the derivative of the sigmoid at the stored probability
__device__ __forceinline__ float4 dsigmoid4(const float4& o, const float4& p) {
    return make_float4(o.x * ((1.0f - p.x) * p.x), o.y * ((1.0f - p.y) * p.y), o.z * ((1.0f - p.z) * p.z),
                       o.w * ((1.0f - p.w) * p.w));
}

struct BoxCursor {
    uint32_t slot, addr, parity;  // ring position, shared address of that slot, parity of the fill waited for
};

// LOGITS: the tensor holds the decoder's pre-activations; phase A turns each element into p = sigmoid(l) once and
// writes it back into its shared-memory slot, phase B reads p and chains the sigmoid's derivative into the result.
template <bool BINARY, bool LOGITS, int INNER4, int NBOX>
__device__ __forceinline__ void boxf_phase_a(BoxCursor& cur, uint32_t slots_u, uint32_t slot_bytes, uint32_t nslot,
                                             uint32_t full_u, uint32_t empty_u, uint32_t row_a, uint32_t row_b,
                                             uint32_t x_u, int lane, bool release, float& acc_a, float& acc_b,
                                             float (&rng)[4]) {
    constexpr int VIT = (INNER4 + 31) / 32, XB = INNER4 * NBOX * 16;  // XB: bytes of one x array
#pragma unroll
    for (int q = 0; q < NBOX; ++q) {
        mbar_wait_u32(full_u + cur.slot * 8, cur.parity);
#pragma unroll
        for (int i = 0; i < VIT; ++i) {
            if ((i + 1) * 32 <= INNER4 || lane + 32 * i < INNER4) {
                const uint32_t o = (uint32_t)(i * 512);
                float4 pa = lds128_u32(cur.addr + row_a + o), pb = lds128_u32(cur.addr + row_b + o);
                if (LOGITS) {
                    pa = sigmoid4(pa);
                    pb = sigmoid4(pb);
                    sts128_u32(cur.addr + row_a + o, pa);
                    sts128_u32(cur.addr + row_b + o, pb);
                }
                const uint32_t xo = x_u + (uint32_t)(q * INNER4 * 16) + o;
                if (BINARY) {
                    const float4 c = lds128_u32(xo), e = lds128_u32(xo + XB);
                    {
                        const float t0 = (pa.x - c.x) + e.x, t1 = (pa.y - c.y) + e.y, t2 = (pa.z - c.z) + e.z,
                                    t3 = (pa.w - c.w) + e.w;
                        acc_a += fast_log2(fabsf((t0 * t1) * (t2 * t3)));
                        rng[0] = fminf(rng[0], fminf(pa.x, pa.y));
                        rng[0] = fminf(rng[0], fminf(pa.z, pa.w));
                        rng[1] = fmaxf(rng[1], fmaxf(pa.x, pa.y));
                        rng[1] = fmaxf(rng[1], fmaxf(pa.z, pa.w));
                    }
                    {
                        const float t0 = (pb.x - c.x) + e.x, t1 = (pb.y - c.y) + e.y, t2 = (pb.z - c.z) + e.z,
                                    t3 = (pb.w - c.w) + e.w;
                        acc_b += fast_log2(fabsf((t0 * t1) * (t2 * t3)));
                        rng[2] = fminf(rng[2], fminf(pb.x, pb.y));
                        rng[2] = fminf(rng[2], fminf(pb.z, pb.w));
                        rng[3] = fmaxf(rng[3], fmaxf(pb.x, pb.y));
                        rng[3] = fmaxf(rng[3], fmaxf(pb.z, pb.w));
                    }
                } else {
                    const float4 xx = lds128_u32(xo);
                    float mn = 1.0f;
                    acc_a += lpmf4<false>(pa, xx, mn);
                    acc_b += lpmf4<false>(pb, xx, mn);
                }
            }
        }
        if (release) {  // forward only: the box is dead after its first read
            if (LOGITS) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane == 0) mbar_arrive_u32(empty_u + cur.slot * 8);
        }
        cur.addr += slot_bytes;
        if (++cur.slot == nslot) { cur.slot = 0; cur.addr = slots_u; cur.parity ^= 1u; }
    }
}

template <bool BINARY, bool LOGITS, int INNER4, int NBOX>
__device__ __forceinline__ void boxf_phase_b(uint32_t bs, uint32_t bs_addr, uint32_t slots_u, uint32_t slot_bytes,
                                             uint32_t nslot, uint32_t empty_u, uint32_t row_a, uint32_t row_b,
                                             uint32_t x_u, int lane, float ga, float gb, float* __restrict__ da,
                                             float* __restrict__ db, bool has_b) {
    constexpr int VIT = (INNER4 + 31) / 32, XB = INNER4 * NBOX * 16;
#pragma unroll
    for (int q = 0; q < NBOX; ++q) {
#pragma unroll
        for (int i = 0; i < VIT; ++i) {
            if ((i + 1) * 32 <= INNER4 || lane + 32 * i < INNER4) {
                const uint32_t o = (uint32_t)(i * 512);
                const float4 pa = lds128_u32(bs_addr + row_a + o), pb = lds128_u32(bs_addr + row_b + o);
                const uint32_t xo = x_u + (uint32_t)(q * INNER4 * 16) + o;
                float4 oa, ob;
                if (BINARY) {
                    const float4 c = lds128_u32(xo), e = lds128_u32(xo + XB);
                    oa.x = ga * fast_rcp((pa.x - c.x) + e.x);
                    oa.y = ga * fast_rcp((pa.y - c.y) + e.y);
                    oa.z = ga * fast_rcp((pa.z - c.z) + e.z);
                    oa.w = ga * fast_rcp((pa.w - c.w) + e.w);
                    ob.x = gb * fast_rcp((pb.x - c.x) + e.x);
                    ob.y = gb * fast_rcp((pb.y - c.y) + e.y);
                    ob.z = gb * fast_rcp((pb.z - c.z) + e.z);
                    ob.w = gb * fast_rcp((pb.w - c.w) + e.w);
                } else {
                    const float4 xx = lds128_u32(xo);
                    oa = dprobs4<false>(pa, xx, ga);
                    ob = dprobs4<false>(pb, xx, gb);
                }
                if (LOGITS) {
                    oa = dsigmoid4(oa, pa);
                    ob = dsigmoid4(ob, pb);
                }
                stg_hint(da + q * INNER4 * 4 + i * 128, oa, 0);
                if (has_b) stg_hint(db + q * INNER4 * 4 + i * 128, ob, 0);
            }
        }
        // LOGITS: this warp's generic-proxy writes to the slot (phase A) precede the async-proxy refill
        if (LOGITS) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive_u32(empty_u + bs * 8);
        bs_addr += slot_bytes;
        if (++bs == nslot) { bs = 0; bs_addr = slots_u; }
    }
}

// Poisson likelihood (zhusuan/distributions/poisson.py:75): log p(x | r) = sum_x (xlogy(x, r) - r) - C_b.  The stager
// stages the raw counts and C_b = sum_x lgamma(x + 1) once per column (it shifts every log-weight of the column by the
// same amount: no weight and no gradient depends on it); the row warps add x log2(r) -- skipped where x == 0, which is
// most elements of count data -- and r separately.
// log(k!) for k < 32: counts are mostly small integers, and lgammaf on the stager's single warp (a long dependent
// chain per element) otherwise sets the column period
__constant__ float c_log_factorial[32] = {
    0.000000000e+00f, 0.000000000e+00f, 6.931471806e-01f, 1.791759469e+00f,
    3.178053830e+00f, 4.787491743e+00f, 6.579251212e+00f, 8.525161361e+00f,
    1.060460290e+01f, 1.280182748e+01f, 1.510441257e+01f, 1.750230785e+01f,
    1.998721450e+01f, 2.255216385e+01f, 2.519122118e+01f, 2.789927138e+01f,
    3.067186011e+01f, 3.350507345e+01f, 3.639544521e+01f, 3.933988419e+01f,
    4.233561646e+01f, 4.538013890e+01f, 4.847118135e+01f, 5.160667557e+01f,
    5.478472940e+01f, 5.800360522e+01f, 6.126170176e+01f, 6.455753863e+01f,
    6.788974314e+01f, 7.125703897e+01f, 7.465823635e+01f, 7.809222355e+01f};
__device__ __forceinline__ float lgamma1p_count(float v) {
    return (v >= 0.f && v < 32.f && v == truncf(v)) ? c_log_factorial[(int)v] : lgammaf(v + 1.f);
}
__device__ __forceinline__ void stage_x_poisson(float* s_xrow, int* s_cb, const float* __restrict__ xrow, int X4, int lane) {
    const float4* src = reinterpret_cast<const float4*>(xrow);
    float4* dst = reinterpret_cast<float4*>(s_xrow);
    float c = 0.f;
    for (int v = lane; v < X4; v += 32) {
        const float4 t = __ldg(src + v);
        dst[v] = t;
        c += (lgamma1p_count(t.x) + lgamma1p_count(t.y)) + (lgamma1p_count(t.z) + lgamma1p_count(t.w));
    }
    c = warp_sum(c);
    if (lane == 0) *s_cb = __float_as_int(c);
}
// The Poisson row loops use the SFU's log2 and reciprocal WITHOUT flush-to-zero: a subnormal rate (exp(l) for a decoder
// output l < -87.3) with a positive count has a finite x log r in torch and in the two-pass route's logf, where the
// .ftz forms would read it as 0 and give -inf (a NaN column when every particle does so).
__device__ __forceinline__ float log2_approx_sub(float x) {
    float y;
    asm("lg2.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx_sub(float x) {
    float y;
    asm("rcp.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float xlog2(float x, float r) { return x == 0.f ? 0.f : x * log2_approx_sub(r); }

template <int INNER4, int NBOX>
__device__ __forceinline__ void boxf_phase_a_poisson(BoxCursor& cur, uint32_t slots_u, uint32_t slot_bytes, uint32_t nslot,
                                                     uint32_t full_u, uint32_t empty_u, uint32_t row_a, uint32_t row_b,
                                                     uint32_t x_u, int lane, bool release, float& acc_a, float& acc_b,
                                                     float& rsum_a, float& rsum_b) {
    constexpr int VIT = (INNER4 + 31) / 32;
#pragma unroll
    for (int q = 0; q < NBOX; ++q) {
        mbar_wait_u32(full_u + cur.slot * 8, cur.parity);
#pragma unroll
        for (int i = 0; i < VIT; ++i) {
            if ((i + 1) * 32 <= INNER4 || lane + 32 * i < INNER4) {
                const uint32_t o = (uint32_t)(i * 512);
                const float4 pa = lds128_u32(cur.addr + row_a + o), pb = lds128_u32(cur.addr + row_b + o);
                const float4 xx = lds128_u32(x_u + (uint32_t)(q * INNER4 * 16) + o);
                acc_a += (xlog2(xx.x, pa.x) + xlog2(xx.y, pa.y)) + (xlog2(xx.z, pa.z) + xlog2(xx.w, pa.w));
                acc_b += (xlog2(xx.x, pb.x) + xlog2(xx.y, pb.y)) + (xlog2(xx.z, pb.z) + xlog2(xx.w, pb.w));
                rsum_a += (pa.x + pa.y) + (pa.z + pa.w);
                rsum_b += (pb.x + pb.y) + (pb.z + pb.w);
            }
        }
        if (release) {  // forward only: the box is dead after its first read
            __syncwarp();
            if (lane == 0) mbar_arrive_u32(empty_u + cur.slot * 8);
        }
        cur.addr += slot_bytes;
        if (++cur.slot == nslot) { cur.slot = 0; cur.addr = slots_u; cur.parity ^= 1u; }
    }
}

// drate = g (x / r - 1) = (g x) rcp(r) - g
__device__ __forceinline__ float4 drate4(const float4& r, const float4& xx, float g) {
    return make_float4(fmaf(g * xx.x, rcp_approx_sub(r.x), -g), fmaf(g * xx.y, rcp_approx_sub(r.y), -g),
                       fmaf(g * xx.z, rcp_approx_sub(r.z), -g), fmaf(g * xx.w, rcp_approx_sub(r.w), -g));
}

template <int INNER4, int NBOX>
__device__ __forceinline__ void boxf_phase_b_poisson(uint32_t bs, uint32_t bs_addr, uint32_t slots_u, uint32_t slot_bytes,
                                                     uint32_t nslot, uint32_t empty_u, uint32_t row_a, uint32_t row_b,
                                                     uint32_t x_u, int lane, float ga, float gb, float* __restrict__ da,
                                                     float* __restrict__ db, bool has_b) {
    constexpr int VIT = (INNER4 + 31) / 32;
#pragma unroll
    for (int q = 0; q < NBOX; ++q) {
#pragma unroll
        for (int i = 0; i < VIT; ++i) {
            if ((i + 1) * 32 <= INNER4 || lane + 32 * i < INNER4) {
                const uint32_t o = (uint32_t)(i * 512);
                const float4 pa = lds128_u32(bs_addr + row_a + o), pb = lds128_u32(bs_addr + row_b + o);
                const float4 xx = lds128_u32(x_u + (uint32_t)(q * INNER4 * 16) + o);
                stg_hint(da + q * INNER4 * 4 + i * 128, drate4(pa, xx, ga), 0);
                if (has_b) stg_hint(db + q * INNER4 * 4 + i * 128, drate4(pb, xx, gb), 0);
            }
        }
        __syncwarp();
        if (lane == 0) mbar_arrive_u32(empty_u + bs * 8);
        bs_addr += slot_bytes;
        if (++bs == nslot) { bs = 0; bs_addr = slots_u; }
    }
}

template <int EST, int INNER4, int NBOX, bool LOGITS>
__global__ void __launch_bounds__((BOX_MAX_ROW_WARPS + 4) * 32, 1)
    k_iw_bernoulli_boxf(const __grid_constant__ CUtensorMap probs_map, float* __restrict__ cost,
                        float* __restrict__ dprobs, float* __restrict__ dlogp, float* __restrict__ dlogq,
                        float* __restrict__ logpx_out, const float* __restrict__ x,
                        const float* __restrict__ logp_other, const float* __restrict__ logq, int K, int64_t B,
                        int nslot, float gscale, int stagger_groups, int stagger_cycles, int flags, int64_t ldkb,
                        float* __restrict__ loss_out, unsigned* __restrict__ ticket) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int INNER = INNER4 * 4, X = INNER * NBOX, X4 = X / 4;
    const BoxLayout L(K, X, INNER, nslot);
    const int Kpad = L.Kpad;
    const uint32_t slot_bytes = (uint32_t)L.slot_bytes();
    unsigned char* slots = smem + L.slots_off();
    float* s_x = reinterpret_cast<float*>(smem + L.x_off());
    double* s_xw = reinterpret_cast<double*>(smem + L.xw_off());
    double* s_xv = reinterpret_cast<double*>(smem + L.xv_off());
    float* s_lpx = reinterpret_cast<float*>(smem + L.lpx_off());
    float* s_other = reinterpret_cast<float*>(smem + L.other_off());
    float* s_lq = reinterpret_cast<float*>(smem + L.lq_off());
    int* s_bin = reinterpret_cast<int*>(smem + L.bin_off());
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bar_off());
    uint64_t* empty = full + nslot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // warp roles: [0, NW) row warps | NW stager | NW+1, NW+2 objective warps (even / odd columns) | NW+3 producer
    const int NW = (blockDim.x >> 5) - 4;
    const uint32_t box_bytes = (uint32_t)K * (uint32_t)INNER * 4u;
    const float LN2 = 0.6931471805599453f;
    const int64_t ncols = ((int64_t)blockIdx.x < B) ? (B - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < nslot; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], (uint32_t)NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    auto stage_scalars = [&](int64_t b, int buf) { stage_scalars_batched(s_other + buf * Kpad, s_lq + buf * Kpad, logp_other, logq, K, ldkb, b, lane); };
    auto stage_x = [&](int64_t b, int slot) { stage_x_batched(s_x + (size_t)slot * 2 * X, s_bin + slot, x + b * X, X4, lane); };
    const bool is_stager = warp == NW, is_obj = warp == NW + 1 || warp == NW + 2, is_producer = warp == NW + 3;
    pdl_wait();  // everything above touched shared memory only; probs / x / the [K,B] terms may come from the kernel before
    pdl_trigger();
    stagger_start(stagger_groups, stagger_cycles);
    // Column 0 only: column 1 is staged while column 0 is being read.  The first tensor copies are issued AFTER
    // this staging on purpose: issuing them first (measured here and in the ring kernel: +4 and +7 us per launch)
    // starts every CTA's column 0 at the same instant, and the chip then alternates between a read-only phase A
    // and a write-heavy phase B in lock-step; the variable staging latency spreads the CTAs out.
    if (is_stager && ncols > 0) {
        stage_scalars(blockIdx.x, 0);
        stage_x(blockIdx.x, 0);
    }
    __syncthreads();

    if (is_producer) {
        // box t = (column t / NBOX, piece t % NBOX) goes to slot t % nslot.  probs is read exactly once: its lines
        // are marked evict-first, so that 160 MB of it does not push out of L2 what the launch writes and the
        // kernels around it read.  Measured on one B200: the IWAE step 83.1 -> 78.9 us (profiles/r3_boxf_rows.md)
        if (lane == 0) {
            uint64_t evict_first;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(evict_first));
            int slot = 0, q = 0;
            uint32_t wait_parity = 1;
            bool first_pass = true;
            int64_t col = blockIdx.x;
            const int64_t ntask = ncols * NBOX;
            for (int64_t t = 0; t < ntask; ++t) {
                if (!first_pass) mbar_wait(&empty[slot], wait_parity);
                mbar_expect_tx(&full[slot], box_bytes);
                tma_load_box_hint(slots + (size_t)slot * slot_bytes, &probs_map, q * INNER, (int)col, 0, &full[slot],
                                  evict_first);
                if (++q == NBOX) { q = 0; col += gridDim.x; }
                if (++slot == nslot) {
                    slot = 0;
                    if (first_pass) { first_pass = false; wait_parity = 0; }
                    else wait_parity ^= 1u;
                }
            }
        }
        return;
    }
    const int sync_threads = (NW + 2) * 32;
    if (is_stager) {
        int64_t b = blockIdx.x;
        if (ncols > 1) {
            stage_scalars(b + gridDim.x, 1);
            stage_x(b + gridDim.x, 1);
        }
        for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
            named_bar_sync(1 + (int)(c & 1), sync_threads);
            if (c + 2 < ncols) {
                stage_scalars(b + 2 * (int64_t)gridDim.x, (int)((c + 2) & 3));
                stage_x(b + 2 * (int64_t)gridDim.x, (int)((c + 2) % 3));
            }
        }
        return;
    }
    if (is_obj) {
        const int p = warp - NW - 1;
        int64_t b = (int64_t)blockIdx.x + (int64_t)p * gridDim.x;
        double part = 0.0;
        for (int64_t c = p; c < ncols; c += 2, b += 2 * (int64_t)gridDim.x) {
            const int buf = (int)(c & 3);
            named_bar_sync(1 + p, sync_threads);
            part += (double)column_objective<EST>(lane, K, ldkb, b, s_lpx + buf * Kpad, s_other + buf * Kpad,
                                                  s_lq + buf * Kpad, s_xw + p * Kpad, gscale, cost, dlogp, dlogq,
                                                  logpx_out, flags);
        }
        finish_loss(lane, p, part, loss_out, ticket);
        return;
    }

    // ---- row warps: rows ka = warp and kb = warp + NW of every column (kb may not exist) ----------------
    const int ka = warp, kb = warp + NW;
    const bool has_b = kb < K;
    const int kb_eff = has_b ? kb : ka;
    const uint32_t slots_u = smem_u32(slots), full_u = smem_u32(full), empty_u = smem_u32(empty);
    const uint32_t row_a = (uint32_t)ka * (INNER * 4) + (uint32_t)lane * 16, row_b = (uint32_t)kb_eff * (INNER * 4) + (uint32_t)lane * 16;
    const uint32_t sx_u = smem_u32(s_x) + (uint32_t)lane * 16;
    BoxCursor cur{0u, slots_u, 0u};
    int64_t b = blockIdx.x;
    for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
        const int par = (int)(c & 3), xs = (int)(c % 3);
        const uint32_t x_u = sx_u + (uint32_t)xs * (2 * X * 4);
        // the stager publishes column 1's x only after the first rendezvous of column 0 for c >= 2; column 1's
        // staging is ordered by the rendezvous of column 0 as well (the stager arrives after staging it)
        const bool binary = s_bin[xs] != 0;
        const uint32_t slot0 = cur.slot, addr0 = cur.addr;
        float acc_a = 0.f, acc_b = 0.f;
        float rng[4] = {0.f, 0.f, 0.f, 0.f};
        if (binary)
            boxf_phase_a<true, LOGITS, INNER4, NBOX>(cur, slots_u, slot_bytes, (uint32_t)nslot, full_u, empty_u, row_a, row_b, x_u,
                                             lane, dprobs == nullptr, acc_a, acc_b, rng);
        else
            boxf_phase_a<false, LOGITS, INNER4, NBOX>(cur, slots_u, slot_bytes, (uint32_t)nslot, full_u, empty_u, row_a, row_b, x_u,
                                              lane, dprobs == nullptr, acc_a, acc_b, rng);
        if (binary) {
            if (rng[0] < -1e-8f || rng[1] > 1.0f) acc_a = __int_as_float(0x7fc00000);
            if (rng[2] < -1e-8f || rng[3] > 1.0f) acc_b = __int_as_float(0x7fc00000);
        }
        acc_a = warp_sum(acc_a);
        acc_b = warp_sum(acc_b);
        if (lane == 0) {
            const float la = acc_a * LN2;
            s_lpx[par * Kpad + ka] = la;
            s_xv[par * Kpad + ka] = ((double)la - (double)s_lq[par * Kpad + ka]) + (double)s_other[par * Kpad + ka];
            if (has_b) {
                const float lb = acc_b * LN2;
                s_lpx[par * Kpad + kb] = lb;
                s_xv[par * Kpad + kb] = ((double)lb - (double)s_lq[par * Kpad + kb]) + (double)s_other[par * Kpad + kb];
            }
        }
        named_bar_sync(1 + (int)(c & 1), sync_threads);
        if (dprobs) {
            double m1;
            float invS;
            ring_max_sumexp(lane, K, s_xv + par * Kpad, m1, invS);
            const float ga = -(expf((float)(s_xv[par * Kpad + ka] - m1)) * invS) * gscale;
            const float gb = -(expf((float)(s_xv[par * Kpad + kb_eff] - m1)) * invS) * gscale;
            float* da = dprobs + ((int64_t)ka * B + b) * X + lane * 4;
            float* db = dprobs + ((int64_t)kb_eff * B + b) * X + lane * 4;
            if (binary)
                boxf_phase_b<true, LOGITS, INNER4, NBOX>(slot0, addr0, slots_u, slot_bytes, (uint32_t)nslot, empty_u, row_a, row_b, x_u,
                                                 lane, ga, gb, da, db, has_b);
            else
                boxf_phase_b<false, LOGITS, INNER4, NBOX>(slot0, addr0, slots_u, slot_bytes, (uint32_t)nslot, empty_u, row_a, row_b, x_u,
                                                  lane, ga, gb, da, db, has_b);
        }
    }
}

// Poisson likelihood over rates [K,B,X] (zs_iw_poisson_fused): the roles, barriers, staging pipeline and objective of
// k_iw_bernoulli_boxf with the Poisson stager and row loops above; `probs_map` maps the rates, `dprobs` receives drate.
// A kernel of its own rather than a likelihood parameter of k_iw_bernoulli_boxf: routing both through one inlined body
// changed the register allocation of the Bernoulli instantiations, which stay as they were.
template <int EST, int INNER4, int NBOX>
__global__ void __launch_bounds__((BOX_MAX_ROW_WARPS + 4) * 32, 1)
    k_iw_poisson_boxf(const __grid_constant__ CUtensorMap probs_map, float* __restrict__ cost,
                      float* __restrict__ dprobs, float* __restrict__ dlogp, float* __restrict__ dlogq,
                      float* __restrict__ logpx_out, const float* __restrict__ x,
                      const float* __restrict__ logp_other, const float* __restrict__ logq, int K, int64_t B,
                      int nslot, float gscale, int stagger_groups, int stagger_cycles, int flags, int64_t ldkb,
                      float* __restrict__ loss_out, unsigned* __restrict__ ticket) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int INNER = INNER4 * 4, X = INNER * NBOX, X4 = X / 4;
    const BoxLayout L(K, X, INNER, nslot);
    const int Kpad = L.Kpad;
    const uint32_t slot_bytes = (uint32_t)L.slot_bytes();
    unsigned char* slots = smem + L.slots_off();
    float* s_x = reinterpret_cast<float*>(smem + L.x_off());
    double* s_xw = reinterpret_cast<double*>(smem + L.xw_off());
    double* s_xv = reinterpret_cast<double*>(smem + L.xv_off());
    float* s_lpx = reinterpret_cast<float*>(smem + L.lpx_off());
    float* s_other = reinterpret_cast<float*>(smem + L.other_off());
    float* s_lq = reinterpret_cast<float*>(smem + L.lq_off());
    int* s_bin = reinterpret_cast<int*>(smem + L.bin_off());
    uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.bar_off());
    uint64_t* empty = full + nslot;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // warp roles: [0, NW) row warps | NW stager | NW+1, NW+2 objective warps (even / odd columns) | NW+3 producer
    const int NW = (blockDim.x >> 5) - 4;
    const uint32_t box_bytes = (uint32_t)K * (uint32_t)INNER * 4u;
    const float LN2 = 0.6931471805599453f;
    const int64_t ncols = ((int64_t)blockIdx.x < B) ? (B - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < nslot; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], (uint32_t)NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    auto stage_scalars = [&](int64_t b, int buf) { stage_scalars_batched(s_other + buf * Kpad, s_lq + buf * Kpad, logp_other, logq, K, ldkb, b, lane); };
    // s_bin[slot] holds the bits of the column's C_b (the Bernoulli kernel keeps its binary-x flag there)
    auto stage_x = [&](int64_t b, int slot) { stage_x_poisson(s_x + (size_t)slot * 2 * X, s_bin + slot, x + b * X, X4, lane); };
    const bool is_stager = warp == NW, is_obj = warp == NW + 1 || warp == NW + 2, is_producer = warp == NW + 3;
    pdl_wait();  // everything above touched shared memory only; probs / x / the [K,B] terms may come from the kernel before
    pdl_trigger();
    stagger_start(stagger_groups, stagger_cycles);
    // Column 0 only: column 1 is staged while column 0 is being read.  The first tensor copies are issued AFTER
    // this staging on purpose: issuing them first (measured here and in the ring kernel: +4 and +7 us per launch)
    // starts every CTA's column 0 at the same instant, and the chip then alternates between a read-only phase A
    // and a write-heavy phase B in lock-step; the variable staging latency spreads the CTAs out.
    if (is_stager && ncols > 0) {
        stage_scalars(blockIdx.x, 0);
        stage_x(blockIdx.x, 0);
    }
    __syncthreads();

    if (is_producer) {
        // box t = (column t / NBOX, piece t % NBOX) goes to slot t % nslot
        if (lane == 0) {
            int slot = 0, q = 0;
            uint32_t wait_parity = 1;
            bool first_pass = true;
            int64_t col = blockIdx.x;
            const int64_t ntask = ncols * NBOX;
            for (int64_t t = 0; t < ntask; ++t) {
                if (!first_pass) mbar_wait(&empty[slot], wait_parity);
                mbar_expect_tx(&full[slot], box_bytes);
                tma_load_box(slots + (size_t)slot * slot_bytes, &probs_map, q * INNER, (int)col, 0, &full[slot]);
                if (++q == NBOX) { q = 0; col += gridDim.x; }
                if (++slot == nslot) {
                    slot = 0;
                    if (first_pass) { first_pass = false; wait_parity = 0; }
                    else wait_parity ^= 1u;
                }
            }
        }
        return;
    }
    const int sync_threads = (NW + 2) * 32;
    if (is_stager) {
        int64_t b = blockIdx.x;
        if (ncols > 1) {
            stage_scalars(b + gridDim.x, 1);
            stage_x(b + gridDim.x, 1);
        }
        for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
            named_bar_sync(1 + (int)(c & 1), sync_threads);
            if (c + 2 < ncols) {
                stage_scalars(b + 2 * (int64_t)gridDim.x, (int)((c + 2) & 3));
                stage_x(b + 2 * (int64_t)gridDim.x, (int)((c + 2) % 3));
            }
        }
        return;
    }
    if (is_obj) {
        const int p = warp - NW - 1;
        int64_t b = (int64_t)blockIdx.x + (int64_t)p * gridDim.x;
        double part = 0.0;
        for (int64_t c = p; c < ncols; c += 2, b += 2 * (int64_t)gridDim.x) {
            const int buf = (int)(c & 3);
            named_bar_sync(1 + p, sync_threads);
            part += (double)column_objective<EST>(lane, K, ldkb, b, s_lpx + buf * Kpad, s_other + buf * Kpad,
                                                  s_lq + buf * Kpad, s_xw + p * Kpad, gscale, cost, dlogp, dlogq,
                                                  logpx_out, flags);
        }
        finish_loss(lane, p, part, loss_out, ticket);
        return;
    }

    // ---- row warps: rows ka = warp and kb = warp + NW of every column (kb may not exist) ----------------
    const int ka = warp, kb = warp + NW;
    const bool has_b = kb < K;
    const int kb_eff = has_b ? kb : ka;
    const uint32_t slots_u = smem_u32(slots), full_u = smem_u32(full), empty_u = smem_u32(empty);
    const uint32_t row_a = (uint32_t)ka * (INNER * 4) + (uint32_t)lane * 16, row_b = (uint32_t)kb_eff * (INNER * 4) + (uint32_t)lane * 16;
    const uint32_t sx_u = smem_u32(s_x) + (uint32_t)lane * 16;
    BoxCursor cur{0u, slots_u, 0u};
    int64_t b = blockIdx.x;
    for (int64_t c = 0; c < ncols; ++c, b += gridDim.x) {
        const int par = (int)(c & 3), xs = (int)(c % 3);
        const uint32_t x_u = sx_u + (uint32_t)xs * (2 * X * 4);
        // the stager publishes column 1's x only after the first rendezvous of column 0 for c >= 2; column 1's
        // staging is ordered by the rendezvous of column 0 as well (the stager arrives after staging it)
        const uint32_t slot0 = cur.slot, addr0 = cur.addr;
        const float cb = __int_as_float(s_bin[xs]);
        float acc_a = 0.f, acc_b = 0.f, rsum_a = 0.f, rsum_b = 0.f;
        boxf_phase_a_poisson<INNER4, NBOX>(cur, slots_u, slot_bytes, (uint32_t)nslot, full_u, empty_u, row_a, row_b,
                                           x_u, lane, dprobs == nullptr, acc_a, acc_b, rsum_a, rsum_b);
        acc_a = warp_sum(acc_a);
        acc_b = warp_sum(acc_b);
        rsum_a = warp_sum(rsum_a);
        rsum_b = warp_sum(rsum_b);
        if (lane == 0) {
            const float la = (acc_a * LN2 - rsum_a) - cb;
            s_lpx[par * Kpad + ka] = la;
            s_xv[par * Kpad + ka] = ((double)la - (double)s_lq[par * Kpad + ka]) + (double)s_other[par * Kpad + ka];
            if (has_b) {
                const float lb = (acc_b * LN2 - rsum_b) - cb;
                s_lpx[par * Kpad + kb] = lb;
                s_xv[par * Kpad + kb] = ((double)lb - (double)s_lq[par * Kpad + kb]) + (double)s_other[par * Kpad + kb];
            }
        }
        named_bar_sync(1 + (int)(c & 1), sync_threads);
        if (dprobs) {
            double m1;
            float invS;
            ring_max_sumexp(lane, K, s_xv + par * Kpad, m1, invS);
            const float ga = -(expf((float)(s_xv[par * Kpad + ka] - m1)) * invS) * gscale;
            const float gb = -(expf((float)(s_xv[par * Kpad + kb_eff] - m1)) * invS) * gscale;
            float* da = dprobs + ((int64_t)ka * B + b) * X + lane * 4;
            float* db = dprobs + ((int64_t)kb_eff * B + b) * X + lane * 4;
            boxf_phase_b_poisson<INNER4, NBOX>(slot0, addr0, slots_u, slot_bytes, (uint32_t)nslot, empty_u, row_a,
                                               row_b, x_u, lane, ga, gb, da, db, has_b);
        }
    }
}

static int pick_warps_ring(int K) {
    // row warps (three more warps stage inputs and compute the objective); equal rows per warp if possible
    for (int d = ZS_RING_MAX_ROW_WARPS; d >= 4; --d)
        if (K % d == 0) return d;
    return K < 24 ? (K < 1 ? 1 : K) : 24;
}

}  // namespace zs

using namespace zs;

namespace {

long long* g_trace = nullptr;  // zs_debug_set_trace
int g_impl_override = -1;      // zs_debug_set_fused_impl

enum { IMPL_RING = 2, IMPL_BOX = 3, IMPL_BOXG = 4 };

// Developer knobs, read from the environment ONCE per process (the hot path never calls getenv):
//   ZS_FUSED_IMPL       ring | box (default: fixed-geometry box kernels where instantiated, else the generic box kernel,
//                       else the ring) | boxg (generic box kernel only); zs_debug_set_fused_impl overrides at run time
//   ZS_FUSED_GRID       fewer CTAs than SMs (per-SM vs chip-level bound)
//   ZS_FUSED_STAGGER    "groups,cycles" of the CTA start stagger
//   ZS_FUSED_L2_AHEAD   boxes requested into L2 ahead of the shared-memory copies (generic box kernel)
//   ZS_FUSED_RING_DEPTH slots per row warp of the ring kernel;  ZS_FUSED_EARLY  first bulk copies before the staging
struct FusedKnobs {
    int impl = IMPL_BOX, grid_cap = 0, l2_ahead = 0, ring_depth = 4, early = ZS_RING_EARLY_DEFAULT;
    bool stagger_set = false;
    int stagger_groups = 0, stagger_cycles = 0;
    FusedKnobs() {
        if (const char* e = getenv("ZS_FUSED_IMPL")) {
            if (e[0] == 'r') impl = IMPL_RING;
            else if (e[0] == 'b') impl = (e[1] == 'o' && e[2] == 'x' && e[3] == 'g') ? IMPL_BOXG : IMPL_BOX;
        }
        if (const char* e = getenv("ZS_FUSED_GRID")) grid_cap = atoi(e);
        if (const char* e = getenv("ZS_FUSED_L2_AHEAD")) l2_ahead = atoi(e);
        if (const char* e = getenv("ZS_FUSED_RING_DEPTH")) ring_depth = atoi(e) < 1 ? 1 : atoi(e);
        if (const char* e = getenv("ZS_FUSED_EARLY"))
            if (e[0] != 0) early = e[0] != '0';
        if (const char* e = getenv("ZS_FUSED_STAGGER"))
            stagger_set = sscanf(e, "%d%*c%d", &stagger_groups, &stagger_cycles) == 2;  // "2,4000" or "2x4000"
    }
};
const FusedKnobs& knobs() {
    static const FusedKnobs k;
    return k;
}
int fused_impl_choice() { return g_impl_override >= 0 ? g_impl_override : knobs().impl; }

// One fused launch, as the internal launchers see it.  The [K, .] arrays (logp_other, logq, dlogp, dlogq,
// logpx_out) have row pitch `ldkb` >= B: the host-buffer step runs chunks of columns straight out of / into
// full-size device arrays.
struct FusedCall {
    int estimator;
    float *cost, *dprobs, *dlogp, *dlogq, *logpx_out;
    const float *probs, *x, *logp_other, *logq;
    int64_t K, B, X, ldkb;
    double grad_scale;
    int kflags;  // FUSED_ACCUMULATE | FUSED_EARLY_ISSUE, as the kernels read them
    bool logits;
    cudaStream_t st;
    float* loss_out = nullptr;   // sum_b cost[b], written by the launch itself (finish_loss), or null
    unsigned* ticket = nullptr;  // its workspace: counter word + per-warp partial sums (finish_loss)
    bool poisson = false;        // `probs` holds Poisson rates, `x` counts (zs_iw_poisson_fused)
};

// Tensor map of probs[K][B][X] with box {inner, 1, K}; the driver's encoder is looked up through the runtime.
typedef CUresult (*zs_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int make_probs_map(CUtensorMap* map, const float* probs, int64_t K, int64_t B, int64_t X, int inner) {
    static zs_encode_tiled_fn encode = nullptr;
    if (encode == nullptr) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult qres;
        ZS_CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
        if (fn == nullptr || qres != cudaDriverEntryPointSuccess) {
            set_last_error_msg("cuTensorMapEncodeTiled is not available in this driver");
            return ZS_ERR_UNSUPPORTED;
        }
        encode = (zs_encode_tiled_fn)fn;
    }
    const cuuint64_t dims[3] = {(cuuint64_t)X, (cuuint64_t)B, (cuuint64_t)K};
    const cuuint64_t strides[2] = {(cuuint64_t)X * 4, (cuuint64_t)B * (cuuint64_t)X * 4};
    const cuuint32_t box[3] = {(cuuint32_t)inner, 1, (cuuint32_t)K};
    const cuuint32_t estr[3] = {1, 1, 1};
    const CUresult r = encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(probs), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_last_error_msg("cuTensorMapEncodeTiled rejected the probs layout");
        return ZS_ERR_UNSUPPORTED;
    }
    return ZS_OK;
}

// Box geometry: `inner` divides X, is a multiple of 4 and at most 256 floats (the copy engine's box limit);
// the best choice keeps the most lanes busy (inner/4 float4 per row piece against 32-lane steps).
int pick_box_inner(int64_t X) {
    int best = 0;
    double best_eff = 0.0;
    for (int inner = 256; inner >= 32; inner -= 4) {
        if (X % inner != 0) continue;
        const int f4 = inner / 4;
        const double eff = (double)f4 / (32.0 * ((f4 + 31) / 32));
        if (eff > best_eff + 1e-9) { best_eff = eff; best = inner; }
    }
    return best_eff >= 0.7 ? best : 0;
}

struct Stagger {
    int groups, cycles;
};
// Start-time stagger of the persistent CTAs (stagger_start).
Stagger pick_stagger(int64_t K, int64_t X, int64_t B, int64_t grid) {
    if (knobs().stagger_set) return Stagger{knobs().stagger_groups, knobs().stagger_cycles};
    if (grid <= 1 || B < 4 * grid) return Stagger{1, 0};  // fewer than four columns per CTA: nothing to desynchronise
    // measured at K=50, X=784 (column period ~16k cycles): 3-6 groups spanning 4000-5000 cycles are all within
    // 1% of each other (66.7 us against 70.5 us without); 4 groups of K*X/26 cycles
    const int64_t cyc = K * X / 26;
    return Stagger{4, (int)(cyc > 10000 ? 10000 : cyc)};
}

int max_optin_smem(int* out) {
    static int cached_dev = -1, cached = 0;
    int dev = 0;
    ZS_CUDA_TRY(cudaGetDevice(&dev));
    if (dev != cached_dev) {
        ZS_CUDA_TRY(cudaDeviceGetAttribute(&cached, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        cached_dev = dev;
    }
    *out = cached;
    return ZS_OK;
}

int64_t persistent_grid(int64_t B) {
    int64_t grid = sm_count();
    if (knobs().grid_cap > 0 && grid > knobs().grid_cap) grid = knobs().grid_cap;
    return grid > B ? B : grid;
}

int launch_fused_box(const FusedCall& c, bool generic_only) {
    const int64_t K = c.K, B = c.B, X = c.X;
    if (K > 2 * BOX_MAX_ROW_WARPS || B >= ((int64_t)1 << 31) || X * 4 % 16 != 0) {
        set_last_error_msg("box kernel: at most two rows per warp (K <= 50)");
        return ZS_ERR_UNSUPPORTED;
    }
    const int inner = pick_box_inner(X);
    if (inner == 0) {
        set_last_error_msg("box kernel: no box width divides X well");
        return ZS_ERR_UNSUPPORTED;
    }
    int max_optin = 0;
    int rc = max_optin_smem(&max_optin);
    if (rc != ZS_OK) return rc;
    const int nbox = (int)(X / inner);
    int nslot = 2 * nbox;  // at most a whole column of prefetch
    while (nslot > nbox && BoxLayout((int)K, (int)X, inner, nslot).total() > (size_t)max_optin) --nslot;
    if (nslot < nbox + 1 || BoxLayout((int)K, (int)X, inner, nslot).total() > (size_t)max_optin) {
        set_last_error_msg("box kernel: a column plus one box does not fit in shared memory");
        return ZS_ERR_UNSUPPORTED;
    }
    CUtensorMap map;
    rc = make_probs_map(&map, c.probs, K, B, X, inner);
    if (rc != ZS_OK) return rc;
    const int nw = K <= BOX_MAX_ROW_WARPS ? (int)K : (int)((K + 1) / 2);
    const size_t smem = BoxLayout((int)K, (int)X, inner, nslot).total();
    const int threads = (nw + 4) * 32;
    const int64_t grid = persistent_grid(B);
    const Stagger stg = pick_stagger(K, X, B, grid);
    // fixed-geometry instantiations (fully unrolled box loops) for the common row lengths
    using boxf_fn = decltype(&k_iw_bernoulli_boxf<ZS_EST_SGVB, 28, 7, false>);
    boxf_fn fixed = nullptr;
    if (!generic_only) {
        const bool sg = c.estimator == ZS_EST_SGVB;
#define ZS_BOXF_PICK(I4, NB)                                                                                        \
    if (inner == 4 * (I4) && nbox == (NB))                                                                           \
        fixed = c.poisson ? (sg ? k_iw_poisson_boxf<ZS_EST_SGVB, I4, NB> : k_iw_poisson_boxf<ZS_EST_VIMCO, I4, NB>)      \
              : c.logits  ? (sg ? k_iw_bernoulli_boxf<ZS_EST_SGVB, I4, NB, true> : k_iw_bernoulli_boxf<ZS_EST_VIMCO, I4, NB, true>) \
                          : (sg ? k_iw_bernoulli_boxf<ZS_EST_SGVB, I4, NB, false> : k_iw_bernoulli_boxf<ZS_EST_VIMCO, I4, NB, false>)
        ZS_BOXF_PICK(28, 7);   // X = 784
        ZS_BOXF_PICK(32, 1);   // X = 128
        ZS_BOXF_PICK(64, 1);   // X = 256
        ZS_BOXF_PICK(64, 2);   // X = 512
        ZS_BOXF_PICK(64, 4);   // X = 1024
#undef ZS_BOXF_PICK
    }
    if (fixed != nullptr) {
        // Bernoulli at K <= 25: two rows per row warp as well, not one row per warp (whose row b repeats row a and is
        // dropped): the warp's x load serves two rows.  Measured on one B200 at K = 25, B = 1024, X = 784:
        // 47.7 -> 37.7 us (profiles/r3_boxf_rows.md)
        const int nw_fixed = c.poisson ? nw : (int)((K + 1) / 2);
        ZS_CUDA_TRY(cudaFuncSetAttribute(fixed, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        launch_pdl(PDL_FUSED, fixed, dim3((unsigned)grid), dim3((nw_fixed + 4) * 32), smem, c.st, map, c.cost, c.dprobs, c.dlogp, c.dlogq,
                   c.logpx_out, c.x, c.logp_other, c.logq, (int)K, B, nslot, (float)c.grad_scale, stg.groups, stg.cycles,
                   c.kflags, c.ldkb, c.loss_out, c.ticket);
        ZS_LAUNCH_CHECK(c.poisson ? "k_iw_poisson_boxf" : "k_iw_bernoulli_boxf");
        return ZS_OK;
    }
    if (c.logits || c.poisson) {
        set_last_error_msg(c.poisson ? "fused Poisson step: no fixed-geometry kernel instantiated for this row length"
                                     : "fused logits form: no fixed-geometry kernel instantiated for this row length");
        return ZS_ERR_UNSUPPORTED;
    }
    auto kern = c.estimator == ZS_EST_SGVB ? k_iw_bernoulli_box<ZS_EST_SGVB> : k_iw_bernoulli_box<ZS_EST_VIMCO>;
    ZS_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // boxes requested into L2 ahead of the shared-memory copies: measured no gain (0..4) to a loss (>= 7), off
    kern<<<(unsigned)grid, threads, smem, c.st>>>(map, c.cost, c.dprobs, c.dlogp, c.dlogq, c.logpx_out, c.x, c.logp_other,
                                                  c.logq, (int)K, B, (int)X, inner, nslot, knobs().l2_ahead,
                                                  (float)c.grad_scale, stg.groups, stg.cycles, c.kflags, g_trace, c.ldkb,
                                                  c.loss_out, c.ticket);
    ZS_LAUNCH_CHECK("k_iw_bernoulli_box");
    return ZS_OK;
}

int launch_fused_ring(const FusedCall& c) {
    const int64_t K = c.K, B = c.B, X = c.X;
    if (c.logits || c.poisson) {
        set_last_error_msg("fused logits / Poisson form: only the fixed-geometry box kernels take it");
        return ZS_ERR_UNSUPPORTED;
    }
    int max_optin = 0;
    int rc = max_optin_smem(&max_optin);
    if (rc != ZS_OK) return rc;
    // per-warp mini-rings: NW row warps x D slots each; deepest D (<= 4) that fits, fewer warps if needed
    int nw = pick_warps_ring((int)K);
    int D = knobs().ring_depth;
    while (D > 1 && RingLayout((int)K, (int)X, nw * D).total() > (size_t)max_optin) --D;
    while (nw > 1 && RingLayout((int)K, (int)X, nw * D).total() > (size_t)max_optin) --nw;
    if (RingLayout((int)K, (int)X, nw * D).total() > (size_t)max_optin) {
        set_last_error_msg("ring kernel: a row slot does not fit in shared memory");
        return ZS_ERR_UNSUPPORTED;
    }
    const int R = nw * D;
    const size_t smem = RingLayout((int)K, (int)X, R).total();
    const int threads = (nw + 3) * 32;
    const bool sgvb = c.estimator == ZS_EST_SGVB;
    const int trips = ((int)(X / 4) + 31) / 32;  // 128-bit loads per lane and row
    // exact trip counts of common row lengths are fully unrolled (784 -> 7)
    auto kern = sgvb ? k_iw_bernoulli_ring<ZS_EST_SGVB, 0> : k_iw_bernoulli_ring<ZS_EST_VIMCO, 0>;
    switch (trips) {
        case 2: kern = sgvb ? k_iw_bernoulli_ring<ZS_EST_SGVB, 2> : k_iw_bernoulli_ring<ZS_EST_VIMCO, 2>; break;
        case 4: kern = sgvb ? k_iw_bernoulli_ring<ZS_EST_SGVB, 4> : k_iw_bernoulli_ring<ZS_EST_VIMCO, 4>; break;
        case 7: kern = sgvb ? k_iw_bernoulli_ring<ZS_EST_SGVB, 7> : k_iw_bernoulli_ring<ZS_EST_VIMCO, 7>; break;
        case 8: kern = sgvb ? k_iw_bernoulli_ring<ZS_EST_SGVB, 8> : k_iw_bernoulli_ring<ZS_EST_VIMCO, 8>; break;
        default: break;
    }
    ZS_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t grid = persistent_grid(B);
    const Stagger stg = pick_stagger(K, X, B, grid);
    kern<<<(unsigned)grid, threads, smem, c.st>>>(c.cost, c.dprobs, c.dlogp, c.dlogq, c.logpx_out, c.probs, c.x,
                                                  c.logp_other, c.logq, (int)K, B, (int)X, R, (float)c.grad_scale,
                                                  stg.groups, stg.cycles,
                                                  c.kflags | (knobs().early ? FUSED_EARLY_ISSUE : 0), g_trace, c.ldkb,
                                                  c.loss_out, c.ticket);
    ZS_LAUNCH_CHECK("k_iw_bernoulli_ring");
    return ZS_OK;
}

// fixed-geometry box kernel -> generic box kernel -> row-streaming ring; ZS_ERR_UNSUPPORTED / ZS_ERR_ALIGN when no
// fused kernel takes the shape (the caller composes the two-pass entry points)
int fused_launch(const FusedCall& c) {
    if (c.X % 4 != 0 || c.K > 4096 || c.X > (1 << 20)) {
        set_last_error_msg("fused kernel needs X % 4 == 0 and K <= 4096");
        return ZS_ERR_UNSUPPORTED;
    }
    if (!aligned16(c.probs) || !aligned16(c.x) || !aligned16(c.dprobs)) {
        set_last_error_msg("fused kernel needs 16-byte aligned probs / x / dprobs");
        return ZS_ERR_ALIGN;
    }
    const int impl = fused_impl_choice();
    if (impl >= IMPL_BOX) {
        const int rc = launch_fused_box(c, impl == IMPL_BOXG);
        if (rc != ZS_ERR_UNSUPPORTED) return rc;
    }
    return launch_fused_ring(c);
}

// The checks and the FusedCall of the four fused entry points.  `with_loss`: the _loss form, which also writes the
// mean objective and so needs loss_out, workspace, cost, at least one column and a grid its workspace covers.
int fused_entry(bool poisson, bool with_loss, int estimator, float* loss_out, void* workspace, float* cost,
                float* dprobs, float* dlogp, float* dlogq, float* logpx_out, const float* probs, const float* x,
                const float* logp_other, const float* logq, int64_t K, int64_t B, int64_t X, double grad_scale,
                int flags, zs_stream_t stream) {
    ZS_REQUIRE(probs && x && K >= 1 && B >= 0 && X >= 1, ZS_ERR_ARG);
    ZS_REQUIRE(!with_loss || (loss_out && workspace && cost && B >= 1), ZS_ERR_ARG);
    ZS_REQUIRE(estimator == ZS_EST_SGVB || estimator == ZS_EST_VIMCO, ZS_ERR_ARG);
    ZS_REQUIRE(!(estimator == ZS_EST_VIMCO && (K < 2 || logq == nullptr)), ZS_ERR_ARG);
    const int allowed = ZS_FUSED_ACCUMULATE_COST | ZS_FUSED_COST_SCALED | (poisson ? 0 : ZS_FUSED_LOGITS);
    ZS_REQUIRE((flags & ~allowed) == 0, ZS_ERR_ARG);
    if (B == 0) return ZS_OK;
    if (with_loss) ZS_REQUIRE(persistent_grid(B) <= ZS_FUSED_LOSS_MAX_GRID, ZS_ERR_UNSUPPORTED);
    FusedCall c{estimator, cost, dprobs, dlogp, dlogq, logpx_out, probs, x, logp_other, logq, K, B, X, B, grad_scale,
                ((flags & ZS_FUSED_ACCUMULATE_COST) ? FUSED_ACCUMULATE : 0) |
                    ((flags & ZS_FUSED_COST_SCALED) ? FUSED_COST_SCALED : 0),
                (flags & ZS_FUSED_LOGITS) != 0,
                as_stream(stream),
                loss_out,
                (unsigned*)workspace,
                poisson};
    return fused_launch(c);
}

}  // namespace

extern "C" {

int zs_iw_bernoulli_fused(int estimator, float* cost, float* dprobs, float* dlogp, float* dlogq, float* logpx_out,
                          const float* probs, const float* x, const float* logp_other, const float* logq, int64_t K,
                          int64_t B, int64_t X, double grad_scale, int flags, zs_stream_t stream) {
    return fused_entry(false, false, estimator, nullptr, nullptr, cost, dprobs, dlogp, dlogq, logpx_out, probs, x,
                       logp_other, logq, K, B, X, grad_scale, flags, stream);
}

int zs_iw_bernoulli_fused_loss(int estimator, float* loss_out, void* workspace, float* cost, float* dprobs, float* dlogp,
                               float* dlogq, float* logpx_out, const float* probs, const float* x,
                               const float* logp_other, const float* logq, int64_t K, int64_t B, int64_t X,
                               double grad_scale, int flags, zs_stream_t stream) {
    return fused_entry(false, true, estimator, loss_out, workspace, cost, dprobs, dlogp, dlogq, logpx_out, probs, x,
                       logp_other, logq, K, B, X, grad_scale, flags, stream);
}

int zs_iw_poisson_fused(int estimator, float* cost, float* drate, float* dlogp, float* dlogq, float* logpx_out,
                        const float* rate, const float* x, const float* logp_other, const float* logq, int64_t K,
                        int64_t B, int64_t X, double grad_scale, int flags, zs_stream_t stream) {
    return fused_entry(true, false, estimator, nullptr, nullptr, cost, drate, dlogp, dlogq, logpx_out, rate, x,
                       logp_other, logq, K, B, X, grad_scale, flags, stream);
}

int zs_iw_poisson_fused_loss(int estimator, float* loss_out, void* workspace, float* cost, float* drate, float* dlogp,
                             float* dlogq, float* logpx_out, const float* rate, const float* x, const float* logp_other,
                             const float* logq, int64_t K, int64_t B, int64_t X, double grad_scale, int flags,
                             zs_stream_t stream) {
    return fused_entry(true, true, estimator, loss_out, workspace, cost, drate, dlogp, dlogq, logpx_out, rate, x,
                       logp_other, logq, K, B, X, grad_scale, flags, stream);
}

/* Debug hooks (not used by the Python package's hot path). */
int zs_debug_set_trace(void* device_buffer) {
    g_trace = (long long*)device_buffer;
    return ZS_OK;
}
int zs_debug_set_fused_impl(int impl) {
    ZS_REQUIRE(impl == -1 || impl == IMPL_RING || impl == IMPL_BOX || impl == IMPL_BOXG, ZS_ERR_ARG);
    g_impl_override = impl;
    return ZS_OK;
}

}  // extern "C"

// ---- host-buffer step, pipelined over column chunks -----------------------------------------------
// Batch columns are independent, so the step is cut into chunks of columns that flow through the handle's
// streams: H2D copy of chunk c+1, fused kernel on chunk c and D2H copy of chunk c-1 overlap (PCIe is
// full duplex), with HS_NBUF rotating device buffers.  The [K,B,X] host layout is gathered / scattered
// with 2-D copies (K rows of chunk*X floats, host pitch B*X).  The first H2D and the last D2H cannot
// overlap anything; a schedule that starts and ends with small chunks (ZS_HS_CHUNK_MIN=32: 32, 64, 128, ..., 64, 32)
// was measured SLOWER than uniform 128-column chunks (4.06 vs 3.93 ms; 256: 4.14, 512: 4.74; floor 3.45-3.5 ms):
// the K = 50 strided rows of a small chunk are short DMA segments.  Uniform chunks are the default.
// The small results (cost, dlogp, dlogq) travel on their own stream ahead of the big dprobs copies, so
// a caller can go on (zs_iw_step_host_wait(h, 0)) while the gradient of the likelihood is still landing.
// All state lives in the caller's handle (zs_host_step_create): any number of handles may be in flight, one step
// per handle at a time.
namespace {
constexpr int HS_NBUF = 3;
constexpr int HS_MAX_CHUNKS = 4096;
// columns per chunk (ZS_HS_CHUNK) and the size of the first / last chunk (ZS_HS_CHUNK_MIN): dev knobs, read once
int64_t hs_env(const char* name, int64_t dflt) {
    const char* e = getenv(name);
    const long v = e ? atol(e) : 0;
    return v > 0 ? (int64_t)v : dflt;
}
const int64_t HS_CHUNK = hs_env("ZS_HS_CHUNK", 128);
const int64_t HS_CHUNK_MIN = hs_env("ZS_HS_CHUNK_MIN", 128);
inline int64_t up256(int64_t v) { return (v + 255) & ~(int64_t)255; }
}  // namespace

struct zs_host_step {
    int device = -1;
    cudaStream_t s_in = nullptr, s_run = nullptr, s_out = nullptr, s_small = nullptr;
    cudaEvent_t ev_in[HS_NBUF] = {}, ev_run[HS_NBUF] = {}, ev_out[HS_NBUF] = {}, ev_start = nullptr;
    cudaEvent_t ev_small_done = nullptr, ev_all_done = nullptr;
    bool pending = false;
    int64_t sizes[HS_MAX_CHUNKS];
};

namespace {
// chunk sizes: HS_CHUNK_MIN, 2 HS_CHUNK_MIN, ... at the head and mirrored at the tail, HS_CHUNK in between
int chunk_schedule(int64_t B, int64_t* sizes) {
    int n = 0;
    int64_t head[8], tail[8];
    int nh = 0, nt = 0;
    int64_t left = B;
    for (int64_t c = HS_CHUNK_MIN; c < HS_CHUNK && left >= 4 * c; c *= 2) {
        head[nh++] = c;
        tail[nt++] = c;
        left -= 2 * c;
    }
    for (int i = 0; i < nh; ++i) sizes[n++] = head[i];
    while (left > 0 && n < HS_MAX_CHUNKS - 8) {
        const int64_t c = left < HS_CHUNK ? left : HS_CHUNK;
        sizes[n++] = c;
        left -= c;
    }
    if (left > 0) return -1;
    for (int i = nt - 1; i >= 0; --i) sizes[n++] = tail[i];
    return n;
}

// run `body` with the handle's device current
struct DeviceScope {
    int prev = -1, want = -1;
    explicit DeviceScope(int dev) : want(dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != want) cudaSetDevice(want);
    }
    ~DeviceScope() {
        if (prev >= 0 && prev != want) cudaSetDevice(prev);
    }
};
}  // namespace

extern "C" {

int zs_host_step_create(zs_host_step** out) {
    ZS_REQUIRE(out != nullptr, ZS_ERR_ARG);
    *out = nullptr;
    zs_host_step* h = new (std::nothrow) zs_host_step();
    ZS_REQUIRE(h != nullptr, ZS_ERR_ARG);
    auto fail = [&](cudaError_t e, const char* what) {
        set_last_error(what, e);
        zs_host_step_destroy(h);
        return ZS_ERR_CUDA;
    };
    cudaError_t e = cudaGetDevice(&h->device);
    if (e != cudaSuccess) return fail(e, "cudaGetDevice");
    for (cudaStream_t* s : {&h->s_in, &h->s_run, &h->s_out, &h->s_small})
        if ((e = cudaStreamCreateWithFlags(s, cudaStreamNonBlocking)) != cudaSuccess) return fail(e, "cudaStreamCreate");
    for (int i = 0; i < HS_NBUF; ++i)
        for (cudaEvent_t* ev : {&h->ev_in[i], &h->ev_run[i], &h->ev_out[i]})
            if ((e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreate");
    for (cudaEvent_t* ev : {&h->ev_start, &h->ev_small_done, &h->ev_all_done})
        if ((e = cudaEventCreateWithFlags(ev, cudaEventDisableTiming)) != cudaSuccess) return fail(e, "cudaEventCreate");
    *out = h;
    return ZS_OK;
}

int zs_host_step_destroy(zs_host_step* h) {
    if (h == nullptr) return ZS_OK;
    DeviceScope scope(h->device);
    if (h->pending && h->ev_all_done) cudaEventSynchronize(h->ev_all_done);
    for (cudaStream_t s : {h->s_in, h->s_run, h->s_out, h->s_small})
        if (s) cudaStreamDestroy(s);
    for (int i = 0; i < HS_NBUF; ++i)
        for (cudaEvent_t ev : {h->ev_in[i], h->ev_run[i], h->ev_out[i]})
            if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : {h->ev_start, h->ev_small_done, h->ev_all_done})
        if (ev) cudaEventDestroy(ev);
    (void)cudaGetLastError();
    delete h;
    return ZS_OK;
}

int64_t zs_iw_step_host_workspace(int64_t K, int64_t B, int64_t X) {
    if (K < 1 || B < 0 || X < 1) return -1;
    const int64_t c = B < HS_CHUNK ? (B > 0 ? B : 1) : HS_CHUNK;
    const int64_t per = 2 * up256(K * c * X * 4) + up256(c * X * 4) + 5 * up256(K * c * 4) + up256(c * 4);
    // + full-size [K,B] log-weight terms and gradients, and the per-column costs
    return HS_NBUF * per + 4 * up256(K * B * 4) + up256(B * 4);
}

int zs_iw_step_host_wait(zs_host_step* h, int what) {
    ZS_REQUIRE(h != nullptr && (what == 0 || what == 1), ZS_ERR_ARG);
    if (!h->pending) return ZS_OK;
    DeviceScope scope(h->device);
    if (what == 0) {
        ZS_CUDA_TRY(cudaEventSynchronize(h->ev_small_done));
    } else {
        ZS_CUDA_TRY(cudaEventSynchronize(h->ev_all_done));
        h->pending = false;
    }
    return ZS_OK;
}

int zs_iw_step_host_begin(zs_host_step* ctx, int estimator, float* cost_host, float* dprobs_host, float* dlogp,
                          float* dlogq, const float* probs_host, const float* x_host, const float* logp_other,
                          const float* logq, int64_t K, int64_t B, int64_t X, double grad_scale, void* ws,
                          int64_t ws_bytes, int scalars_on_device, zs_stream_t stream) {
    ZS_REQUIRE(ctx && probs_host && x_host && ws && K >= 1 && B >= 1 && X >= 1, ZS_ERR_ARG);
    ZS_REQUIRE(estimator == ZS_EST_SGVB || estimator == ZS_EST_VIMCO, ZS_ERR_ARG);
    ZS_REQUIRE(!(estimator == ZS_EST_VIMCO && logq == nullptr), ZS_ERR_ARG);
    if (ws_bytes < zs_iw_step_host_workspace(K, B, X)) return ZS_ERR_WORKSPACE;
    ZS_REQUIRE(aligned16(ws), ZS_ERR_ALIGN);
    int dev = -1;
    ZS_CUDA_TRY(cudaGetDevice(&dev));
    if (dev != ctx->device) {
        set_last_error_msg("host step: the handle was created on another device");
        return ZS_ERR_ARG;
    }
    int rc = ZS_OK;
    // a previous step of this handle whose big copies were left in flight shares the workspace: let it land first
    if (ctx->pending) {
        rc = zs_iw_step_host_wait(ctx, 1);
        if (rc != ZS_OK) return rc;
    }
    int64_t* sizes = ctx->sizes;
    const int nchunks = chunk_schedule(B, sizes);
    if (nchunks < 0) {
        set_last_error_msg("host step: too many column chunks");
        return ZS_ERR_UNSUPPORTED;
    }
    const int64_t C = B < HS_CHUNK ? B : HS_CHUNK;
    const int64_t kcx = up256(K * C * X * 4), cx = up256(C * X * 4), kc = up256(K * C * 4), cb = up256(C * 4);
    const int64_t per = 2 * kcx + cx + 5 * kc + cb;
    struct Buf {
        float *probs, *dprobs, *x, *other, *logq, *dlogp, *dlogq, *lpx, *cost;
    } buf[HS_NBUF];
    for (int i = 0; i < HS_NBUF; ++i) {
        char* p = (char*)ws + i * per;
        buf[i].probs = (float*)p; p += kcx;
        buf[i].dprobs = (float*)p; p += kcx;
        buf[i].x = (float*)p; p += cx;
        buf[i].other = (float*)p; p += kc;   // the dense [K,bc] arrays serve the two-pass fallback only
        buf[i].logq = (float*)p; p += kc;
        buf[i].dlogp = (float*)p; p += kc;
        buf[i].dlogq = (float*)p; p += kc;
        buf[i].lpx = (float*)p; p += kc;
        buf[i].cost = (float*)p;
    }
    const bool dev_sc = scalars_on_device != 0;
    const int64_t kb = up256(K * B * 4);
    char* gp = (char*)ws + HS_NBUF * per;
    // full-size device arrays of the [K,B] terms: the caller's own (device mode) or workspace copies of the
    // host arrays, moved with ONE contiguous copy each way instead of K short rows per chunk
    float* other_full = dev_sc ? const_cast<float*>(logp_other) : (logp_other ? (float*)gp : nullptr);
    float* logq_full = dev_sc ? const_cast<float*>(logq) : (logq ? (float*)(gp + kb) : nullptr);
    float* dlogp_full = dev_sc ? dlogp : (float*)(gp + 2 * kb);
    float* dlogq_full = dev_sc ? dlogq : (float*)(gp + 3 * kb);
    float* cost_full = (float*)(gp + 4 * kb);
    if (dev_sc && dlogp_full == nullptr) dlogp_full = (float*)(gp + 2 * kb);
    if (dev_sc && dlogq_full == nullptr) dlogq_full = (float*)(gp + 3 * kb);
    // order the internal streams after whatever the caller already enqueued
    ZS_CUDA_TRY(cudaEventRecord(ctx->ev_start, as_stream(stream)));
    ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_in, ctx->ev_start, 0));
    ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_run, ctx->ev_start, 0));
    ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_out, ctx->ev_start, 0));
    ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_small, ctx->ev_start, 0));
    ctx->pending = true;
    if (!dev_sc) {
        if (logp_other)
            ZS_CUDA_TRY(cudaMemcpyAsync(other_full, logp_other, K * B * 4, cudaMemcpyHostToDevice, ctx->s_in));
        if (logq) ZS_CUDA_TRY(cudaMemcpyAsync(logq_full, logq, K * B * 4, cudaMemcpyHostToDevice, ctx->s_in));
    }

    int64_t b0 = 0;
    for (int c = 0; c < nchunks; ++c) {
        const int i = c % HS_NBUF;
        const int64_t bc = sizes[c];
        Buf& d = buf[i];
        // the buffer set is free once the D2H copy of chunk c - HS_NBUF is done
        if (c >= HS_NBUF) ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_in, ctx->ev_out[i], 0));
        ZS_CUDA_TRY(cudaMemcpy2DAsync(d.probs, bc * X * 4, probs_host + b0 * X, B * X * 4, bc * X * 4, K,
                                      cudaMemcpyHostToDevice, ctx->s_in));
        ZS_CUDA_TRY(cudaMemcpyAsync(d.x, x_host + b0 * X, bc * X * 4, cudaMemcpyHostToDevice, ctx->s_in));
        ZS_CUDA_TRY(cudaEventRecord(ctx->ev_in[i], ctx->s_in));

        ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_run, ctx->ev_in[i], 0));
        if (c >= HS_NBUF) ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_run, ctx->ev_out[i], 0));  // dprobs buffer reuse
        zs_stream_t run = (zs_stream_t)ctx->s_run;
        FusedCall call{estimator, cost_full + b0, dprobs_host ? d.dprobs : nullptr, dlogp_full + b0, dlogq_full + b0,
                       nullptr, d.probs, d.x, other_full ? other_full + b0 : nullptr, logq_full ? logq_full + b0 : nullptr,
                       K, bc, X, B, grad_scale, 0, false, ctx->s_run};
        rc = fused_launch(call);
        if (rc == ZS_ERR_UNSUPPORTED || rc == ZS_ERR_ALIGN) {
            // two-pass form on dense [K,bc] copies of the chunk's columns: likelihood log-pmf, objective,
            // likelihood backward
            if (other_full)
                ZS_CUDA_TRY(cudaMemcpy2DAsync(d.other, bc * 4, other_full + b0, B * 4, bc * 4, K, cudaMemcpyDeviceToDevice,
                                              ctx->s_run));
            if (logq_full)
                ZS_CUDA_TRY(cudaMemcpy2DAsync(d.logq, bc * 4, logq_full + b0, B * 4, bc * 4, K, cudaMemcpyDeviceToDevice,
                                              ctx->s_run));
            else
                ZS_CUDA_TRY(cudaMemsetAsync(d.logq, 0, K * bc * 4, ctx->s_run));
            rc = zs_bernoulli_logpmf_fwd(ZS_F32, d.lpx, d.x, ZS_KBCAST, d.probs, ZS_FULL, K, bc, X, run);
            if (rc != ZS_OK) return rc;
            rc = zs_iw_objective(ZS_F32, estimator, cost_full + b0, d.dlogp, d.dlogq, d.lpx, d.logq,
                                 other_full ? d.other : nullptr, K, bc, grad_scale, run);
            if (rc != ZS_OK) return rc;
            if (dprobs_host)
                rc = zs_bernoulli_logpmf_bwd(ZS_F32, nullptr, d.dprobs, d.dlogp, d.x, ZS_KBCAST, d.probs, ZS_FULL, K,
                                             bc, X, run);
            if (rc != ZS_OK) return rc;
            ZS_CUDA_TRY(cudaMemcpy2DAsync(dlogp_full + b0, B * 4, d.dlogp, bc * 4, bc * 4, K, cudaMemcpyDeviceToDevice,
                                          ctx->s_run));
            ZS_CUDA_TRY(cudaMemcpy2DAsync(dlogq_full + b0, B * 4, d.dlogq, bc * 4, bc * 4, K, cudaMemcpyDeviceToDevice,
                                          ctx->s_run));
        }
        if (rc != ZS_OK) return rc;
        ZS_CUDA_TRY(cudaEventRecord(ctx->ev_run[i], ctx->s_run));

        ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_out, ctx->ev_run[i], 0));
        if (dprobs_host)
            ZS_CUDA_TRY(cudaMemcpy2DAsync(dprobs_host + b0 * X, B * X * 4, d.dprobs, bc * X * 4, bc * X * 4, K,
                                          cudaMemcpyDeviceToHost, ctx->s_out));
        ZS_CUDA_TRY(cudaEventRecord(ctx->ev_out[i], ctx->s_out));
        b0 += bc;
    }
    // small results: one contiguous copy each, on their own stream, right after the last kernel (ahead of the
    // tail of the dprobs copies).  "small results landed" also means every kernel has run; "all landed" joins
    // every internal stream.  The caller's stream is ordered after the kernels so device-resident gradients can
    // be consumed from it without a host round trip.
    const int last = (nchunks - 1) % HS_NBUF;
    ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_small, ctx->ev_run[last], 0));
    if (cost_host) ZS_CUDA_TRY(cudaMemcpyAsync(cost_host, cost_full, B * 4, cudaMemcpyDeviceToHost, ctx->s_small));
    if (!dev_sc) {
        if (dlogp) ZS_CUDA_TRY(cudaMemcpyAsync(dlogp, dlogp_full, K * B * 4, cudaMemcpyDeviceToHost, ctx->s_small));
        if (dlogq) ZS_CUDA_TRY(cudaMemcpyAsync(dlogq, dlogq_full, K * B * 4, cudaMemcpyDeviceToHost, ctx->s_small));
    }
    ZS_CUDA_TRY(cudaEventRecord(ctx->ev_small_done, ctx->s_small));
    ZS_CUDA_TRY(cudaStreamWaitEvent(ctx->s_out, ctx->ev_small_done, 0));
    ZS_CUDA_TRY(cudaEventRecord(ctx->ev_all_done, ctx->s_out));
    ZS_CUDA_TRY(cudaStreamWaitEvent(as_stream(stream), ctx->ev_run[last], 0));
    return ZS_OK;
}

int zs_iw_step_host(zs_host_step* h, int estimator, float* cost_host, float* dprobs_host, float* dlogp_host,
                    float* dlogq_host, const float* probs_host, const float* x_host, const float* logp_other_host,
                    const float* logq_host, int64_t K, int64_t B, int64_t X, double grad_scale, void* ws,
                    int64_t ws_bytes, zs_stream_t stream) {
    int rc = zs_iw_step_host_begin(h, estimator, cost_host, dprobs_host, dlogp_host, dlogq_host, probs_host, x_host,
                                   logp_other_host, logq_host, K, B, X, grad_scale, ws, ws_bytes, 0, stream);
    if (rc != ZS_OK) {
        if (h != nullptr) zs_iw_step_host_wait(h, 1);
        return rc;
    }
    return zs_iw_step_host_wait(h, 1);
}

}  // extern "C"
