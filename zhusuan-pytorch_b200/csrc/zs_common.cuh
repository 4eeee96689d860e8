// Shared device/host helpers for the sm_100a stochastic-node kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>

#include "../../include/zs_b200.h"

namespace zs {

// ---- error plumbing -------------------------------------------------------
void set_last_error(const char* where, cudaError_t e);
void set_last_error_msg(const char* msg);

#define ZS_CUDA_TRY(expr)                                  \
    do {                                                   \
        cudaError_t _e = (expr);                           \
        if (_e != cudaSuccess) {                           \
            ::zs::set_last_error(#expr, _e);               \
            return ZS_ERR_CUDA;                            \
        }                                                  \
    } while (0)

#define ZS_LAUNCH_CHECK(name)                              \
    do {                                                   \
        cudaError_t _e = cudaGetLastError();               \
        if (_e != cudaSuccess) {                           \
            ::zs::set_last_error(name, _e);                \
            return ZS_ERR_CUDA;                            \
        }                                                  \
    } while (0)

#define ZS_REQUIRE(cond, code)                             \
    do {                                                   \
        if (!(cond)) {                                     \
            ::zs::set_last_error_msg("requirement failed: " #cond); \
            return (code);                                 \
        }                                                  \
    } while (0)

// Runs the statements with `T` bound to the element type of `dtype`; any other dtype returns ZS_ERR_DTYPE from the
// enclosing entry point.
#define ZS_DTYPE_SWITCH(dtype, ...)                                      \
    if ((dtype) == ZS_F32) {                                             \
        using T = float;                                                 \
        __VA_ARGS__                                                      \
    } else if ((dtype) == ZS_F64) {                                      \
        using T = double;                                                \
        __VA_ARGS__                                                      \
    } else {                                                             \
        ::zs::set_last_error_msg("dtype must be ZS_F32 or ZS_F64");      \
        return ZS_ERR_DTYPE;                                             \
    }

inline bool valid_mode(int m) { return m == ZS_FULL || m == ZS_KBCAST || m == ZS_SCALAR; }
inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
inline cudaStream_t as_stream(zs_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

int sm_count();  // of the current device (cached per device)

// ---- programmatic dependent launch ------------------------------------------------
// The step is a chain of short launches around one long one, and in a replayed CUDA graph every kernel -> kernel edge
// costs ~1.2 us of drain + launch latency (profiles/r2_notes.md).  The chain's own kernels are therefore launched with
// cudaLaunchAttributeProgrammaticStreamSerialization: their CTAs may be scheduled while the previous kernel of the
// stream is still running and park at pdl_wait() (griddepcontrol.wait: returns once every prerequisite grid has
// completed and its memory is visible), which every such kernel executes BEFORE its first global-memory access.
// pdl_trigger() (griddepcontrol.launch_dependents) lets the NEXT kernel do the same.  Both are no-ops for a kernel
// launched the ordinary way, so the kernels behave identically behind a plain <<<>>> launch.  ZS_PDL=0 disables it.
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// ZS_PDL is a bit mask over the launch sites (PDL_* below).  Default: all but the latent backward -- measured with
// tools/step_breakdown.py (profiles/r2_notes.md): a programmatic latent backward directly behind the fused kernel
// costs the step 2 us (its CTAs take over SMs that the fused kernel's tail frees and then sit in front of nothing),
// the other three sites are worth 3 us together.
enum { PDL_LATENT_FWD = 1, PDL_FUSED = 2, PDL_SCALE = 4, PDL_LATENT_BWD = 8 };
int pdl_mask();
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(int site, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                              Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (pdl_mask() & site) ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}

// ---- 16-byte packs ---------------------------------------------------------
template <typename T>
struct alignas(16) Pack {
    static constexpr int N = 16 / sizeof(T);
    T v[N];
};

template <typename T>
__device__ __forceinline__ Pack<T> ld_pack(const T* p) {
    return *reinterpret_cast<const Pack<T>*>(p);
}
// streaming (read-once) load: do not keep the line in L1.  NOT volatile: the compiler must be free
// to hoist and batch these loads (several in flight per warp); a volatile asm pins each load behind
// the previous load's consumers and leaves the kernel latency-bound (profiles/r1_notes.md).
__device__ __forceinline__ Pack<float> ld_pack_stream(const float* p) {
    Pack<float> r;
    asm("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.v[0]), "=f"(r.v[1]), "=f"(r.v[2]), "=f"(r.v[3])
                 : "l"(p));
    return r;
}
__device__ __forceinline__ Pack<double> ld_pack_stream(const double* p) {
    Pack<double> r;
    asm("ld.global.nc.L1::no_allocate.v2.f64 {%0,%1}, [%2];" : "=d"(r.v[0]), "=d"(r.v[1]) : "l"(p));
    return r;
}
template <typename T>
__device__ __forceinline__ void st_pack(T* p, const Pack<T>& v) {
    *reinterpret_cast<Pack<T>*>(p) = v;
}
__device__ __forceinline__ void st_pack_stream(float* p, const Pack<float>& r) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(r.v[0]), "f"(r.v[1]),
                 "f"(r.v[2]), "f"(r.v[3])
                 : "memory");
}
__device__ __forceinline__ void st_pack_stream(double* p, const Pack<double>& r) {
    asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1,%2};" ::"l"(p), "d"(r.v[0]), "d"(r.v[1]) : "memory");
}

// ---- warp / sub-warp reductions -----------------------------------------------
template <int WIDTH, typename T>
__device__ __forceinline__ T group_sum(T v) {
#pragma unroll
    for (int o = WIDTH / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o, WIDTH);
    return v;
}
template <typename T>
__device__ __forceinline__ T warp_sum(T v) {
    return group_sum<32>(v);
}
template <typename T>
__device__ __forceinline__ T warp_max(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// ---- math ------------------------------------------------------------------
// log2 on the SFU (MUFU.LG2).  |abs err| <= 2^-22 on [0.5,2], <= 2 ulp elsewhere.
// The big Bernoulli tensors need two logs per element; a polynomial logf would make the
// kernel issue-bound instead of HBM-bound (DESIGN.md §kernels).
__device__ __forceinline__ float fast_log2(float x) {
    float y;
    asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
// sigmoid on the SFU: ex2 + rcp (relative error ~1e-6 over |l| <= 40; saturates to exactly 0 / 1 beyond, like
// torch.sigmoid in float32)
__device__ __forceinline__ float fast_sigmoid(float l) {
    float e;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(l * -1.4426950408889634f));
    return fast_rcp(1.0f + e);
}

template <typename T>
struct Real;
template <>
struct Real<float> {
    static __device__ __forceinline__ float log(float x) { return logf(x); }
    static __device__ __forceinline__ float exp(float x) { return expf(x); }
    static __device__ __forceinline__ float sqrt(float x) { return sqrtf(x); }
};
template <>
struct Real<double> {
    static __device__ __forceinline__ double log(double x) { return ::log(x); }
    static __device__ __forceinline__ double exp(double x) { return ::exp(x); }
    static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
};

// grid sizing: enough CTAs to fill the machine a few times, never more than the work
inline int grid_for(int64_t work_items, int items_per_block, int max_waves_blocks_per_sm = 32) {
    int64_t need = (work_items + items_per_block - 1) / items_per_block;
    int64_t cap = (int64_t)sm_count() * max_waves_blocks_per_sm;
    if (need < 1) need = 1;
    return (int)(need < cap ? need : cap);
}

}  // namespace zs
