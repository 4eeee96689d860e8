/*
 * zs_b200.h — C ABI of the B200 (sm_100a) stochastic-node hot path.
 *
 * This is the drop-in boundary for ZhuSuan-PyTorch's multi-particle path.  The
 * reference has no FFI of its own (it is pure Python over torch); every entry
 * point below replaces one Python function of the reference, cited as
 * `file:line` relative to the reference tree.  INTEGRATION.md shows the ctypes
 * stub a reference maintainer would add at each of those sites.
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types cross this boundary;
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *     nothing here synchronises (except the `*_host` convenience calls);
 *   - `dtype` is ZS_F32 or ZS_F64 (the reference's log_floating_dtypes,
 *     zhusuan/distributions/utils.py:5); all tensor arguments of one call share it;
 *   - return value: ZS_OK (0) or a negative ZS_ERR_* code; zs_strerror() names
 *     it, zs_last_error() returns the CUDA error string of the calling thread;
 *   - no global mutable state besides that thread-local error string (and the zs_debug_* developer hooks);
 *     calls that need state across launches take a caller-owned handle or device buffer.
 *
 * Tensor layout ("particle rows")
 *   A stochastic node's value is viewed as [K, M, E], contiguous, where
 *     K = n_particles (the reference's leading `n_samples` axis, base.py:138-140),
 *     M = the batch rows that survive the event reduction,
 *     E = the trailing event elements that are summed (group_ndims axes,
 *         base.py:175-176, and trailing reduce_sum_dims, stochastic_tensor.py:164-165).
 *   Each operand carries a layout mode:
 *     ZS_FULL   [K, M, E]   one value per element
 *     ZS_KBCAST [M, E]      broadcast over particles — replaces `.repeat([K,1,..])`
 *                           (normal.py:94-95,115-116; bernoulli.py:75,90)
 *     ZS_SCALAR [1]         one value for everything
 *   Log-prob outputs are [K, M].
 */
#ifndef ZS_B200_H
#define ZS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* 3: zs_allreduce_sum_peer takes (extra_src, extra_index); new: zs_allreduce_sum_nvls, zs_iw_bernoulli_fused_loss,
 *    zs_debug_set_latent_fwd; later additions (compatible): zs_poisson_*, zs_iw_poisson_fused[_loss], zs_beta_sample,
 *    ZS_FAM_BETA of zs_locscale_logprob_fwd/bwd.  2: device-side Philox state, handle-based host step, flags argument of the fused kernel. */
#define ZS_ABI_VERSION 3

typedef void* zs_stream_t; /* cudaStream_t */

enum { ZS_F32 = 0, ZS_F64 = 1 };
enum { ZS_FULL = 0, ZS_KBCAST = 1, ZS_SCALAR = 2 };
enum { ZS_EST_SGVB = 0, ZS_EST_VIMCO = 1, ZS_EST_ELBO = 2 };
/* location-scale families of the zs_locscale_* entry points (ZS_FAM_BETA: the log-density entry points only) */
enum { ZS_FAM_LOGISTIC = 1, ZS_FAM_LAPLACE = 2, ZS_FAM_UNIFORM = 3, ZS_FAM_BETA = 4 };

enum {
    ZS_OK = 0,
    ZS_ERR_ARG = -1,         /* null pointer / negative size / bad enum          */
    ZS_ERR_DTYPE = -2,       /* dtype not ZS_F32 / ZS_F64                        */
    ZS_ERR_CUDA = -3,        /* a CUDA runtime call or launch failed             */
    ZS_ERR_NO_DEVICE = -4,   /* no sm_100 device visible                         */
    ZS_ERR_WORKSPACE = -5,   /* caller workspace too small (see *_workspace())   */
    ZS_ERR_UNSUPPORTED = -6, /* shape outside what this entry point handles      */
    ZS_ERR_ALIGN = -7        /* pointer not aligned as the entry point requires  */
};

/* ---- library info ------------------------------------------------------- */
int zs_abi_version(void);
const char* zs_strerror(int code);
const char* zs_last_error(void);
/* SM count and compute capability of the current device. */
int zs_device_info(int* sm_count, int* cc_major, int* cc_minor);

/* ---- Philox4x32-10 counter RNG ------------------------------------------
 * Element i of a call uses counter (i/4 lo, i/4 hi, offset lo, offset hi), key
 * (seed lo, seed hi), word i%4.  Results do not depend on the launch geometry.
 * Replaces the CPU-side torch.normal / torch.bernoulli + H2D copies at
 * normal.py:104, bernoulli.py:79, SGLD.py:51, SGHMC.py:27,33,34.
 *
 * Graph-safe stream position.  Every sampling entry point takes (seed, offset, rng_state):
 *   rng_state == NULL : the launch draws from Philox(seed, offset) -- a pure function of its arguments (parity
 *                       tests; also what a captured CUDA graph would replay unchanged, i.e. the SAME noise).
 *   rng_state != NULL : a DEVICE zs_rng_state.  The launch draws from Philox(seed, offset + rng_state->offset) and
 *                       advances rng_state->offset by ZS_RNG_TICK once all of its CTAs have read it, so the next
 *                       sampling launch on the stream -- or the next replay of a captured graph -- draws fresh
 *                       noise.  One state per stream of sampling launches (launches that share a state must be
 *                       stream-ordered).  Initialise with zs_rng_state_init (or write {offset, 0, 0} yourself).
 * Entry points whose backward regenerates the forward's noise also take `rng_snapshot` (DEVICE zs_rng_state, may be
 * NULL): it receives the position the forward used; hand it to the backward as its rng_state (read, not advanced). */
#define ZS_RNG_TICK 4
typedef struct zs_rng_state {
    uint64_t offset;    /* added to the by-value offset                                      */
    uint32_t arrivals;  /* CTAs of the current launch that have read `offset` (0 between launches) */
    uint32_t reserved;
} zs_rng_state;
int zs_rng_state_init(void* rng_state, uint64_t offset, zs_stream_t stream);
int zs_philox_uniform(int dtype, void* out, int64_t n, uint64_t seed, uint64_t offset, void* rng_state,
                      zs_stream_t stream);
int zs_philox_normal(int dtype, void* out, int64_t n, double mean, double std, uint64_t seed, uint64_t offset,
                     void* rng_state, zs_stream_t stream);
/* raw 32-bit words (n must be a multiple of 4); used by the bit-exact RNG tests */
int zs_philox_raw(uint32_t* out, int64_t n, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream);

/* ---- Normal stochastic node ----------------------------------------------
 * zs_normal_sample: z[K,N] = mean + std * eps      (Normal._sample, normal.py:89-107)
 *   eps_in  != NULL : injected noise [K,N] (parity mode; replaces torch.normal(0,1,size))
 *   eps_in  == NULL : eps drawn from Philox(seed, offset), Box-Muller
 *   eps_out != NULL : the noise used is also written there
 *   N = M*E elements per particle; mean/std modes ZS_FULL|ZS_KBCAST|ZS_SCALAR.
 * The same call serves the non-reparameterised branch (torch.normal(mean,std),
 * normal.py:101-102): the value is identical, only autograd differs.            */
int zs_normal_sample(int dtype, void* z, const void* mean, int mean_mode, const void* std, int std_mode,
                     const void* eps_in, void* eps_out, int64_t K, int64_t N, uint64_t seed, uint64_t offset,
                     void* rng_state, void* rng_snapshot, zs_stream_t stream);
/* Pathwise gradient of the sample: dmean = sum_k dz, dstd = sum_k dz*eps (sums only
 * over broadcast axes).  eps == NULL regenerates the noise from (seed, offset).
 * dmean / dstd may be NULL.  SCALAR-mode grads are not produced here (host sums).  */
int zs_normal_sample_bwd(int dtype, void* dmean, int mean_mode, void* dstd, int std_mode, const void* dz,
                         const void* eps, int64_t K, int64_t N, uint64_t seed, uint64_t offset,
                         const void* rng_state, zs_stream_t stream);

/* out[K,M] = sum_e ( c - log(std) - 0.5*exp(-2 log std)*(x-mean)^2 )
 * Normal._log_prob (normal.py:109-126) + Distribution.log_prob's group_ndims sum
 * (base.py:175-176) + StochasticTensor's trailing reduce_sum_dims
 * (stochastic_tensor.py:164-165).                                               */
int zs_normal_logprob_fwd(int dtype, void* out, const void* x, int x_mode, const void* mean, int mean_mode,
                          const void* std, int std_mode, int64_t K, int64_t M, int64_t E, zs_stream_t stream);
/* Backward of the above for upstream g[K,M].  Any of dx/dmean/dstd may be NULL.
 * Each gradient has the layout of its operand: FULL is written elementwise, KBCAST
 * is summed over K in-kernel.  SCALAR gradients are not supported (pass NULL; the
 * host expands the operand instead).                                            */
int zs_normal_logprob_bwd(int dtype, void* dx, void* dmean, void* dstd, const void* g, const void* x, int x_mode,
                          const void* mean, int mean_mode, const void* std, int std_mode, int64_t K, int64_t M,
                          int64_t E, zs_stream_t stream);

/* ---- Logistic / Laplace stochastic nodes (SURVEY 8(f)-4), on the Normal node's kernel templates --------------
 * z[K,N] = loc + scale * eps:  Logistic eps = log u - log(1 - u), u ~ U(0,1)  (Logistic._sample,
 * zhusuan/distributions/logistic.py:56-70, reparameterised);  Laplace eps = -sign(u) log1p(-|u|), u ~ U(-1,1)
 * (torch.distributions.Laplace.sample as called by laplace.py:60-76).  u_in != NULL injects the uniforms.
 * _sample_bwd: dloc = sum_k dz, dscale = sum_k dz * eps (KBCAST) or elementwise (FULL), eps regenerated from
 * (seed, offset) or from `u`.
 * _logprob_fwd: out[K,M] = sum_e log p(x; loc, scale):  Logistic -z - 2 softplus(-z) - log(scale), z = (x-loc)/scale
 * (logistic.py:72-83);  Laplace -log(2 scale) - |x - loc| / scale (laplace.py:78-92).  _logprob_bwd: autograd of those.
 * ZS_FAM_UNIFORM (Uniform, zhusuan/distributions/uniform.py:51-83): _sample draws u ~ U[0,1) (torch.rand, :63-66) and
 * returns loc + scale * u (pass loc = low, scale = high - low; or 0 / 1 for the unit draw the reference caches);
 * _logprob_* take loc = LOW and scale = HIGH: -log(high - low) on [low, high), -inf outside
 * (torch.distributions.Uniform.log_prob, :81), d/dlow = g/(high - low), d/dhigh = -g/(high - low), d/dx = 0.
 * ZS_FAM_BETA (Beta, the reference's zhusuan/distributions/beta.py via torch.distributions.Beta): _logprob_* only, with
 * loc = ALPHA and scale = BETA: xlogy(alpha - 1, x) + xlogy(beta - 1, 1 - x) + lgamma(alpha + beta)
 * - (lgamma(alpha) + lgamma(beta)), and torch's autograd of it (dalpha = xlogy(g, x) + g psi(alpha + beta)
 * - g psi(alpha), likewise dbeta with 1 - x; dx = g (alpha - 1) / x - g (beta - 1) / (1 - x)).  Samples: zs_beta_sample. */
int zs_locscale_sample(int dtype, int family, void* z, const void* loc, int loc_mode, const void* scale, int scale_mode,
                       const void* u_in, int64_t K, int64_t N, uint64_t seed, uint64_t offset, void* rng_state,
                       void* rng_snapshot, zs_stream_t stream);
int zs_locscale_sample_bwd(int dtype, int family, void* dloc, int loc_mode, void* dscale, int scale_mode, const void* dz,
                           const void* u, int64_t K, int64_t N, uint64_t seed, uint64_t offset,
                           const void* rng_state, zs_stream_t stream);
int zs_locscale_logprob_fwd(int dtype, int family, void* out, const void* x, int x_mode, const void* loc, int loc_mode,
                            const void* scale, int scale_mode, int64_t K, int64_t M, int64_t E, zs_stream_t stream);
int zs_locscale_logprob_bwd(int dtype, int family, void* dx, void* dloc, void* dscale, const void* g, const void* x,
                            int x_mode, const void* loc, int loc_mode, const void* scale, int scale_mode, int64_t K,
                            int64_t M, int64_t E, zs_stream_t stream);

/* ---- Bernoulli stochastic node -------------------------------------------
 * out[K,N] = (u < probs) as float, u ~ Philox uniform   (Bernoulli._sample,
 * bernoulli.py:72-82); u_in != NULL injects the uniforms (parity mode).         */
int zs_bernoulli_sample(int dtype, void* out, const void* probs, int probs_mode, const void* u_in, int64_t K,
                        int64_t N, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream);
/* out[K,M] = sum_e ( x*log(p+1e-8) + (1-x)*log((1-p)+1e-8) )
 * Bernoulli._log_prob (bernoulli.py:84-95) + the same event sums as above.      */
int zs_bernoulli_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* probs, int probs_mode,
                            int64_t K, int64_t M, int64_t E, zs_stream_t stream);
/* dprobs = g*( x/(p+1e-8) - (1-x)/((1-p)+1e-8) ), dx = g*(log(p+1e-8)-log((1-p)+1e-8)). */
int zs_bernoulli_logpmf_bwd(int dtype, void* dx, void* dprobs, const void* g, const void* x, int x_mode,
                            const void* probs, int probs_mode, int64_t K, int64_t M, int64_t E,
                            zs_stream_t stream);
/* The same log-pmf for a Bernoulli given by LOGITS: probs = sigmoid(logits) (Bernoulli.__init__,
 * bernoulli.py:47-50) is formed in registers, then bernoulli.py:84-95 as above; dlogits = dprobs * p * (1 - p)
 * (autograd of torch.sigmoid).  Replaces the decoder's Sigmoid + its backward (examples' iwae.py:45-46,75):
 * the [K,M,E] tensor makes one HBM trip each way instead of three.                  */
int zs_bernoulli_logits_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* logits, int logits_mode,
                                   int64_t K, int64_t M, int64_t E, zs_stream_t stream);
int zs_bernoulli_logits_logpmf_bwd(int dtype, void* dx, void* dlogits, const void* g, const void* x, int x_mode,
                                   const void* logits, int logits_mode, int64_t K, int64_t M, int64_t E,
                                   zs_stream_t stream);

/* ---- Poisson stochastic node ------------------------------------------------------------------------------
 * The reference's Poisson (zhusuan/distributions/poisson.py) wraps torch.distributions.Poisson; these replace
 * Poisson._sample (:61, torch.distributions.Poisson.sample) and Poisson._log_prob (:75) + the event sums.
 * zs_poisson_sample: out[K,N] = Poisson(rate) counts as float values, rate mode ZS_FULL|ZS_KBCAST|ZS_SCALAR.  Knuth's
 *   product of uniforms for rate < 10, Hormann's transformed rejection (PTRS) for rate >= 10, as ATen's CPU sampler.
 *   Element i takes its uniforms from the Philox groups (counter i | (j << 48), j = 0, 1, ...; at most 64 groups) of
 *   the position (seed, offset [+ rng_state]): independent of the launch geometry.  Needs K*N < 2^48.
 *   Rates are not validated: negative or NaN rates give 0; rate must be finite.                                    */
int zs_poisson_sample(int dtype, void* out, const void* rate, int rate_mode, int64_t K, int64_t N, uint64_t seed,
                      uint64_t offset, void* rng_state, zs_stream_t stream);
/* out[K,M] = sum_e ( xlogy(x, rate) - rate - lgamma(x + 1) )    (poisson.py:75, torch.distributions.Poisson.log_prob) */
int zs_poisson_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* rate, int rate_mode, int64_t K,
                          int64_t M, int64_t E, zs_stream_t stream);
/* drate = g * (x / rate - 1); the count has no gradient.  drate may be NULL (nothing to do).                          */
int zs_poisson_logpmf_bwd(int dtype, void* drate, const void* g, const void* x, int x_mode, const void* rate,
                          int rate_mode, int64_t K, int64_t M, int64_t E, zs_stream_t stream);

/* ---- Beta stochastic node ---------------------------------------------------------------------------------
 * zs_beta_sample: out[K,N] = Beta(alpha, beta) samples; alpha and beta modes ZS_FULL|ZS_KBCAST|ZS_SCALAR.  As torch's
 *   CPU Dirichlet sampler: two Marsaglia-Tsang gamma draws (shape < 1 boosted), in double, G_alpha / (G_alpha +
 *   G_beta) clamped to [smallest normal of the dtype, nextafter(1, 0)].  Element i takes its words from the Philox
 *   groups (counter i | (j << 48), at most 65 groups) of the position (seed, offset [+ rng_state]), as
 *   zs_poisson_sample: independent of the launch geometry.  Needs K*N < 2^48.  Parameters are not validated: an alpha
 *   or beta that is not positive and finite (0, negative, infinite, NaN) gives NaN.  The log-density is
 *   zs_locscale_logprob_fwd/bwd with ZS_FAM_BETA.                                                                */
int zs_beta_sample(int dtype, void* out, const void* alpha, int alpha_mode, const void* beta, int beta_mode, int64_t K,
                   int64_t N, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream);

/* ---- fused latent-node kernels (zs_latent.cu) -------------------------------
 * Forward: z ~ q (Philox or injected noise), log q(z) and log p(z) under the prior, both summed over
 * E, in ONE launch: Normal._sample + Normal._log_prob twice (normal.py:89-126; the variational net's
 * own log-prob and the generator's prior, iwae.py:60-72,102-120), resp. bernoulli.py:72-95.
 *   mean/std (probs): both ZS_FULL or both ZS_KBCAST; prior_* are [M,E] (KBCAST) or NULL
 *   (standard Normal / Bernoulli(0.5)); logq / logp may be NULL.  Needs E % 4 == 0 and 16-byte
 *   aligned tensors, otherwise ZS_ERR_UNSUPPORTED / ZS_ERR_ALIGN (compose the general kernels).      */
int zs_normal_latent_fwd(int dtype, void* z, void* logq, void* logp, const void* mean, int mean_mode, const void* std,
                         int std_mode, const void* prior_mean, const void* prior_std, const void* eps_in, int64_t K,
                         int64_t M, int64_t E, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream);
/* zbits (may be NULL; float32 / KBCAST only, else ZS_ERR_UNSUPPORTED): the sample once more as bits -- one byte per
 * float4 unit of z ([K, M, E/4] bytes, bit q of byte (k, m, j) = z[k, m, 4j+q]).  zs_bernoulli_latent_bwd reads it
 * instead of z when given: 0.5 MB instead of 8 MB at config 3, behind a kernel whose write-back is still draining. */
int zs_bernoulli_latent_fwd(int dtype, void* z, void* logq, void* logp, const void* probs, int probs_mode,
                            const void* prior_probs, const void* u_in, int64_t K, int64_t M, int64_t E, uint64_t seed,
                            uint64_t offset, void* rng_state, void* zbits, zs_stream_t stream);
/* Backward in ONE launch: gradient of  <dlogq, log q> + <dlogp, log p> + <dz_up, z>  wrt the variational
 * parameters: autograd of both log-densities, the decoder's upstream gradient dz_up [K,M,E] (may be
 * NULL) and, if reparameterized, the pathwise backward of the sample (eps recovered as (z-mean)/std),
 * summed over K for KBCAST parameters.  dlogq / dlogp [K,M] may be NULL.                            */
int zs_normal_latent_bwd(int dtype, void* dmean, void* dstd, const void* dlogq, const void* dlogp, const void* dz_up,
                         const void* z, const void* mean, int mean_mode, const void* std, int std_mode,
                         const void* prior_mean, const void* prior_std, int reparameterized, int64_t K, int64_t M,
                         int64_t E, zs_stream_t stream);
int zs_bernoulli_latent_bwd(int dtype, void* dprobs, const void* dlogq, const void* z, const void* probs,
                            int probs_mode, int64_t K, int64_t M, int64_t E, const void* zbits, zs_stream_t stream);

/* ---- Categorical stochastic node (absent from the reference: parity unpinned;
 * API modelled on bernoulli.py, see DESIGN.md) --------------------------------
 * logits [K|1, M, C]; value = class index stored as float/double in x[K,M].     */
int zs_categorical_sample(int dtype, void* out, const void* logits, int logits_mode, const void* u_in, int64_t K,
                          int64_t M, int64_t C, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream);
int zs_categorical_logpmf_fwd(int dtype, void* out, const void* x, int x_mode, const void* logits, int logits_mode,
                              int64_t K, int64_t M, int64_t C, zs_stream_t stream);
int zs_categorical_logpmf_bwd(int dtype, void* dlogits, const void* g, const void* x, int x_mode,
                              const void* logits, int logits_mode, int64_t K, int64_t M, int64_t C,
                              zs_stream_t stream);

/* ---- multi-particle objectives over log-weights [K,B] ----------------------
 * One launch computes the objective AND its gradient wrt logp and logq.
 *   estimator ZS_EST_SGVB : ImportanceWeightedObjective.sgvb + compute_iw_term
 *       (importance_weighted_objective.py:16-25,102-132)
 *   estimator ZS_EST_VIMCO: ImportanceWeightedObjective.vimco (:134-191), the
 *       [B,K,K] leave-one-out tensor replaced by O(K) per-column sums.
 *   estimator ZS_EST_ELBO : ELBO.sgvb (elbo.py:134-161), cost_b = -mean_k(logp - logq)
 *       (zs_iw_objective only).
 * log w = logp - logq (+ logp_extra when not NULL, a second generator term [K,B]).
 * cost[B]   = per-column surrogate cost (cost_b); the scalar loss is mean_b cost_b.
 * dlogp/dlogq [K,B] = d(sum_b cost_b * grad_scale)/d(logp|logq); pass
 *   grad_scale = 1/B_global to get the gradient of the mean.  Either may be NULL. */
int zs_iw_objective(int dtype, int estimator, void* cost, void* dlogp, void* dlogq, const void* logp,
                    const void* logq, const void* logp_extra, int64_t K, int64_t B, double grad_scale,
                    zs_stream_t stream);
/* buf_i[n_i] *= *scale_dev for up to three buffers (buf1 / buf2 may be NULL), a no-op launch when *scale_dev == 1:
 * applies the upstream gradient of the scalar loss to the gradients the fused kernels computed for a unit upstream
 * gradient (dprobs, dlogp, dlogq) without a host synchronisation and, in the usual case, without touching them. */
int zs_scale_inplace(int dtype, void* buf0, int64_t n0, void* buf1, int64_t n1, void* buf2, int64_t n2,
                     const void* scale_dev, zs_stream_t stream);
/* ELBO.reinforce (zhusuan/variational/elbo.py:163-238), the form the examples use: variance reduction with the
 * moving-mean baseline, no user baseline, mean over all N = prod(shape) elements.  One launch of one 8-CTA
 * thread-block cluster: bc = mean(logp - logq); the float32 state is updated IN PLACE on the device exactly as the
 * reference does (:221-224): mm -= (mm - bc)(1 - decay); ++step; mm /= 1 - decay^step; then
 * cost[0] = -mean(logp + (logp - logq - mm) logq), dlogp = -grad_scale, dlogq = -(logp - logq - mm) grad_scale
 * (pass grad_scale = 1/N).  moving_mean [1] float32 and local_step [1] int32 are DEVICE buffers (the module's
 * registered buffers); dlogp / dlogq may be NULL.                                                          */
int zs_reinforce_step(int dtype, void* cost, void* dlogp, void* dlogq, float* moving_mean, int* local_step,
                      const void* logp, const void* logq, int64_t N, double decay, double grad_scale,
                      zs_stream_t stream);

/* out[0] = scale_a * sum(a[0..na)) + scale_b * sum(b[0..nb)), one launch, fixed summation order.  ELBO.sgvb with a flow
 * (zhusuan/variational/elbo.py:155-161) returns -mean(logp - logq) - sum(log_det): with the per-column costs of
 * zs_iw_objective(ZS_EST_ELBO) as `a` (scale_a = 1/B) and the flow's log-determinants as `b` (scale_b = -1) this is the
 * whole reduction; d out / d a_i = scale_a, d out / d b_i = scale_b.                                    */
int zs_combine_sums(int dtype, void* out, const void* a, int64_t na, double scale_a, const void* b, int64_t nb,
                    double scale_b, zs_stream_t stream);
/* log_mean_exp over the leading axis of [K,B] -> [B]   (zhusuan/utils.py:6-21)    */
int zs_log_mean_exp(int dtype, void* out, const void* x, int64_t K, int64_t B, zs_stream_t stream);
/* backward: dx[K,B] = g[B] * softmax_k(x)                                          */
int zs_log_mean_exp_bwd(int dtype, void* dx, const void* g, const void* x, int64_t K, int64_t B,
                        zs_stream_t stream);

/* ---- fused likelihood + objective kernel: Bernoulli likelihood + IW objective, fwd+bwd in one launch --
 * Replaces, for a Bernoulli likelihood node over [K,B,X] probabilities, Bernoulli._log_prob + the event sum
 * (bernoulli.py:84-95, stochastic_tensor.py:160-181), the log-joint sum (importance_weighted_objective.py:66-77),
 * the estimator (:102-191) and the autograd backward of all three.
 * For every batch column b the K particle rows probs[:, b, :] are brought into shared memory ONCE (TMA tensor
 * copies of {inner, 1, K} boxes; persistent warp-specialised CTAs, one per SM), their log-pmf at x[b,:] is
 * reduced, combined with the rest of the log-weight, the estimator weights are formed, and dprobs is produced
 * from the resident rows -- probs is read from HBM once, dprobs written once.
 *   logp_other[K,B] = sum of the other generator log-probs (may be NULL = 0)
 *   logq[K,B]       = variational log-prob (may be NULL = 0 for SGVB; required for VIMCO)
 *   log w = logpx + logp_other - logq
 *   cost[B], dprobs[K,B,X] (may be NULL: forward only), dlogp[K,B] (= gradient wrt every generator log-prob
 *   term), dlogq[K,B]; logpx_out[K,B] optional copy of the likelihood term.
 * Kernel selection (DESIGN.md 3.1): fixed-geometry box kernel for X in {128, 256, 512, 784, 1024} and K <= 50,
 * generic box kernel for other K <= 50, row-streaming ring kernel for any K <= 4096.
 * Requires f32, X % 4 == 0 and 16-byte aligned probs / dprobs / x; otherwise ZS_ERR_UNSUPPORTED / ZS_ERR_ALIGN and
 * the caller uses the two-pass entry points.
 * flags:
 *   ZS_FUSED_ACCUMULATE_COST  cost[b] += cost_b instead of cost[b] = cost_b: a running sum of the per-column
 *       objectives over steps.  A data-parallel training loop reports its scalar objective from this buffer every N
 *       steps (one reduction + one all-reduce per N steps instead of per step; each column has exactly one writer,
 *       so the sum is deterministic).
 *   ZS_FUSED_LOGITS  `probs` holds LOGITS [K,B,X] (Bernoulli(logits=...), bernoulli.py:47-50): the sigmoid is applied
 *       as the rows arrive in shared memory and its derivative is chained into the result, so `dprobs` is the
 *       gradient w.r.t. the decoder's pre-activations.  Available where a fixed-geometry kernel is instantiated
 *       (X in {128, 256, 512, 784, 1024}, K <= 50); otherwise ZS_ERR_UNSUPPORTED and the caller composes
 *       zs_bernoulli_logits_logpmf_fwd -> zs_iw_objective -> zs_bernoulli_logits_logpmf_bwd.
 *   ZS_FUSED_COST_SCALED  cost[b] = cost_b * grad_scale, so that sum_b cost[b] is the (global-batch) mean objective:
 *       one reduction, no separate scaling pass over the per-column costs.                                  */
enum { ZS_FUSED_ACCUMULATE_COST = 1, ZS_FUSED_LOGITS = 2, ZS_FUSED_COST_SCALED = 4 };
int zs_iw_bernoulli_fused(int estimator, float* cost, float* dprobs, float* dlogp, float* dlogq,
                          float* logpx_out, const float* probs, const float* x, const float* logp_other,
                          const float* logq, int64_t K, int64_t B, int64_t X, double grad_scale, int flags,
                          zs_stream_t stream);

/* The same launch, which also writes the objective itself: loss_out[0] = sum_b cost_b of THIS launch (with
 * ZS_FUSED_COST_SCALED the mean objective of importance_weighted_objective.py:128-129 / :190-191, i.e. what the
 * reference returns from forward()), without a reduction launch after it.  Each of the grid's objective warps keeps
 * the double sum of the float-rounded column costs it wrote; the last one to finish adds the per-warp sums in a fixed
 * order while the row warps are still writing the last columns of dprobs.  Bit-reproducible from launch to launch on
 * one device (the order depends only on the grid size).  `workspace`: ZS_FUSED_LOSS_WS_BYTES of device memory,
 * zero-initialised ONCE by the caller and kept per stream (the kernel re-arms it; two launches that may run
 * concurrently need two workspaces).  `cost` must not be NULL.                                                    */
#define ZS_FUSED_LOSS_MAX_GRID 160
#define ZS_FUSED_LOSS_WS_BYTES (8 + 2 * ZS_FUSED_LOSS_MAX_GRID * 8)
int zs_iw_bernoulli_fused_loss(int estimator, float* loss_out, void* workspace, float* cost, float* dprobs,
                               float* dlogp, float* dlogq, float* logpx_out, const float* probs, const float* x,
                               const float* logp_other, const float* logq, int64_t K, int64_t B, int64_t X,
                               double grad_scale, int flags, zs_stream_t stream);

/* The same fused step for a POISSON likelihood over rates [K,B,X] (zhusuan/distributions/poisson.py:75 instead of
 * bernoulli.py:84-95) with counts x[B,X]; same arguments, flags (ZS_FUSED_LOGITS excepted), workspace and results as
 * the Bernoulli pair above, `drate` in place of `dprobs`.  log p(x_b | rate_k) = sum_x (xlogy(x, r) - r) - C_b with
 * C_b = sum_x lgamma(x + 1), formed once per column.  Only the fixed-geometry box kernel takes it: X in {128, 256,
 * 512, 784, 1024}, K <= 50, f32, 16-byte aligned rate / drate / x; otherwise ZS_ERR_UNSUPPORTED / ZS_ERR_ALIGN and
 * the caller composes zs_poisson_logpmf_fwd -> zs_iw_objective -> zs_poisson_logpmf_bwd.                        */
int zs_iw_poisson_fused(int estimator, float* cost, float* drate, float* dlogp, float* dlogq, float* logpx_out,
                        const float* rate, const float* x, const float* logp_other, const float* logq, int64_t K,
                        int64_t B, int64_t X, double grad_scale, int flags, zs_stream_t stream);
int zs_iw_poisson_fused_loss(int estimator, float* loss_out, void* workspace, float* cost, float* drate, float* dlogp,
                             float* dlogq, float* logpx_out, const float* rate, const float* x,
                             const float* logp_other, const float* logq, int64_t K, int64_t B, int64_t X,
                             double grad_scale, int flags, zs_stream_t stream);

/* Debug hooks.  zs_debug_set_trace: device buffer (grid*40 int64) that the generic box / ring kernels fill with
 * clock64() phase timestamps of each CTA's first 8 columns; NULL (default) disables tracing.
 * zs_debug_set_fused_impl: 2 = ring, 3 = box (default order), 4 = generic box only, -1 = back to the default
 * (the ZS_FUSED_IMPL environment variable, read once per process).  Process-wide; tests and tools only. */
int zs_debug_set_trace(void* device_buffer);
int zs_debug_set_fused_impl(int impl);
/* zs_debug_set_latent_fwd: which float32 / KBCAST forward the latent entry points launch: -1 = by shape (default:
 * the row-per-thread kernel for grids several waves deep, the lane-per-unit kernel otherwise), 0 = lane-per-unit,
 * 1 = row-per-thread wherever the shape qualifies (E <= 64).  Process-wide; tests and tools only.          */
int zs_debug_set_latent_fwd(int impl);

/* ---- SG-MCMC updates across parallel chains (one pass) -----------------------
 * w_out receives the updated chain state and may alias w (in place); the reference
 * returns a fresh leaf tensor per step (SGLD.py:52-54), which costs the same bytes.
 * Velocity / preconditioner state (v, aux) is always updated in place.
 * noise != NULL injects the already-scaled Gaussian term (parity mode); otherwise
 * it is drawn from Philox(seed, offset) inside the kernel.
 * SGLD._update (SGLD.py:42-54):  w += 0.5*lr*g + N(0, lr)                          */
int zs_sgld_step(int dtype, void* w_out, const void* w, const void* g, const void* noise, int64_t n, double lr,
                 uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream);
/* PSGLD._update (SGLD.py:67-82): aux = decay*aux + (1-decay) g^2; G = 1/(eps+sqrt(aux));
 * w += 0.5*lr*G*g + N(0, lr*G).  noise_unit != NULL injects UNIT normals.          */
int zs_psgld_step(int dtype, void* w_out, const void* w, void* aux, const void* g, const void* noise_unit, int64_t n,
                  double lr, double decay, double epsilon, uint64_t seed, uint64_t offset, void* rng_state,
                  zs_stream_t stream);
/* SGHMC._update (SGHMC.py:25-56).
 *   zs_sghmc_pre : optional velocity resample v ~ N(0, lr) (resample != 0; v_noise
 *                  injects it) and, for second_order, the half step w += 0.5 v.
 *   zs_sghmc_post: first order  v = (1-alpha) v + lr g + n ; w += v
 *                  second order v = d (d v + lr g + n), d = exp(-alpha/2) ; w += 0.5 v
 *                  n ~ N(0, 2(alpha-beta) lr) (noise injects it).                   */
int zs_sghmc_pre(int dtype, void* w_out, const void* w, void* v, const void* v_noise, int64_t n, double lr,
                 int resample, int second_order, uint64_t seed, uint64_t offset, void* rng_state, zs_stream_t stream);
int zs_sghmc_post(int dtype, void* w_out, const void* w, void* v, const void* g, const void* noise, int64_t n,
                  double lr, double alpha, double beta, int second_order, uint64_t seed, uint64_t offset,
                  void* rng_state, zs_stream_t stream);

/* Multi-tensor apply: the update of EVERY chain-state tensor of a sampler in ONE launch (the reference loops over
 * the latents in Python, SGLD.py:49-54, SGHMC.py:29-56: one CPU noise draw + H2D + 3-6 kernels each).  The table is
 * read on the host and travels in the kernel parameters, so the call is CUDA-graph capturable and needs no device
 * allocation.  Tensor t owns the quads [q_t, q_t + ceil(n_t / 4)) of ONE Philox stream position (q_0 = 0): element i
 * of tensor t draws word i % 4 of counter q_t + i / 4, so a one-tensor call equals the single-tensor entry point
 * bit for bit, and the whole update consumes one tick.
 *   algorithm ZS_ALG_SGLD       : zs_sgld_step;        state unused
 *             ZS_ALG_PSGLD      : zs_psgld_step;       state = aux, a = decay, b = epsilon, noise = unit normals
 *             ZS_ALG_SGHMC_PRE  : zs_sghmc_pre;        state = v, g unused, noise = injected resampled velocity
 *             ZS_ALG_SGHMC_POST : zs_sghmc_post;       state = v, a = alpha, b = beta
 * At most ZS_CHAIN_MAX_TENSORS tensors per call (ZS_ERR_UNSUPPORTED beyond; split the call). */
#define ZS_CHAIN_MAX_TENSORS 32
enum { ZS_ALG_SGLD = 0, ZS_ALG_PSGLD = 1, ZS_ALG_SGHMC_PRE = 2, ZS_ALG_SGHMC_POST = 3 };
typedef struct zs_chain_tensor {
    void* w_out;       /* updated chain state (may alias w)                          */
    const void* w;     /* current chain state                                         */
    const void* g;     /* gradient of the log joint                                   */
    void* state;       /* v (SGHMC) / aux (PSGLD), updated in place; NULL for SGLD    */
    const void* noise; /* injected noise (parity mode) or NULL = Philox in registers */
    int64_t n;         /* elements                                                    */
} zs_chain_tensor;
int zs_sgmcmc_multi_step(int dtype, int algorithm, const zs_chain_tensor* tensors_host, int n_tensors, double lr,
                         double a, double b, int resample, int second_order, uint64_t seed, uint64_t offset,
                         void* rng_state, zs_stream_t stream);

/* ---- peer-memory all-reduce over NVLink / NVSwitch (zs_collective.cu) ------------------------------------
 * The exchange of the data-parallel path (SURVEY.md 8(e)): SUM of a float32 buffer -- the replicated networks'
 * parameter gradients and the scalar objective -- over the ranks of one node.  The reference has no counterpart
 * (a user would call torch.distributed.all_reduce); for a buffer of a few MB that call is bound by NCCL's launch and
 * protocol latency, so the exchange is a kernel of this library instead:
 *   bufs_host[p]  : base pointer of rank p's buffer as mapped into THIS process (peer / symmetric memory; the same
 *                   layout on every rank), p < world <= ZS_MAX_PEERS
 *   flags_host[p] : rank p's flag area, zs_allreduce_peer_flag_bytes() bytes, zero-initialised before the first call
 *   [first, first + count) : the floats to reduce (multiples of 4); every rank passes the same values
 *   flag_set      : 0 .. ZS_PEER_FLAG_SETS-1; calls that may be in flight at the same time use different sets
 *   ctas          : CTAs of the launch, the same on every rank (0 = default)
 *   extra_src, extra_index : optional device scalar (the step's objective) that this rank's kernel stores into its own
 *                   buffer at float index extra_index (inside [first, first + count)) before the exchange, so the
 *                   caller needs no copy launch to put it there; NULL = nothing
 * Rank r reduces slice r in rank order and stores the sums into every rank's buffer: results are bit-identical on all
 * ranks.  Enqueued on `stream`; every rank must enqueue the matching call (a CTA waits for its counterpart on every
 * peer).  The per-CTA epochs live in the flag area, so the launch can be captured in a CUDA graph and replayed. */
#define ZS_MAX_PEERS 8
#define ZS_PEER_MAX_CTAS 64
#define ZS_PEER_FLAG_SETS 4
#define ZS_PEER_THREADS 512
int64_t zs_allreduce_peer_flag_bytes(void);
int zs_allreduce_sum_peer(float* const* bufs_host, void* const* flags_host, int rank, int world, int64_t first,
                          int64_t count, int flag_set, int ctas, const float* extra_src, int64_t extra_index,
                          zs_stream_t stream);
/* The same exchange through an NVSwitch multicast mapping (NVLS): `multicast_buf` is ONE address that names the buffer
 * in every rank's memory (cuMulticast* / torch symmetric memory's multicast_ptr).  Rank r reads slice r with
 * multimem.ld_reduce (the switch returns the SUM over the ranks) and writes it back with multimem.st (the switch
 * stores into every rank's copy): (1 + 1/N) buffer volumes per GPU and direction instead of 2(N-1)/N.  Flags as above
 * (unicast peer pointers); `local_buf` is this rank's ordinary pointer to its own buffer (for extra_src).  All ranks
 * receive the same bits; the switch's summation order is its own.                                                */
int zs_allreduce_sum_nvls(float* multicast_buf, float* local_buf, void* const* flags_host, int rank, int world,
                          int64_t first, int64_t count, int flag_set, int ctas, const float* extra_src,
                          int64_t extra_index, zs_stream_t stream);

/* ---- host-buffer step (end-to-end measurement, INTEGRATION.md) ----
 * One importance-weighted step of the Bernoulli-likelihood path with HOST buffers for the big
 * tensors (pinned memory recommended): what a caller whose decoder output lives in host memory
 * would hand to ImportanceWeightedObjective.forward + backward
 * (zhusuan/variational/importance_weighted_objective.py:79-132 with the likelihood node of
 * zhusuan/distributions/bernoulli.py:84-95).  Batch columns are independent, so the step is pipelined
 * over chunks of 128 columns on the handle's streams: the H2D copy of chunk c+1, the
 * fused kernel (or the two-pass kernels) on chunk c and the D2H copy of chunk c-1 overlap, so the call
 * costs about max(H2D, D2H) instead of their sum.  `ws` is a caller-owned device workspace of
 * zs_iw_step_host_workspace() bytes (three chunk-sized buffer sets).
 *
 * All state (four streams, the events, the chunk schedule, "a step is in flight") lives in an opaque handle created
 * on the current device: the library keeps no global state for these calls.  Handles are independent (one per
 * thread / per caller stream is fine); one step per handle is in flight at a time, a second _begin on the same handle
 * first waits for the previous step to land.
 *
 *   zs_iw_step_host        ordered after prior work on `stream`; returns after everything has landed.
 *   zs_iw_step_host_begin  enqueues the same step and returns.  With scalars_on_device != 0 the [K,B]
 *                          arrays logp_other / logq / dlogp / dlogq are DEVICE pointers (row pitch B):
 *                          they are gathered / scattered per chunk on the device and `stream` is made
 *                          to wait for the last kernel, so the caller can consume dlogp / dlogq from
 *                          `stream` with no host round trip.  cost / dprobs are always host buffers.
 *   zs_iw_step_host_wait   what = 0: the small results (cost; host dlogp / dlogq) have landed and every
 *                          kernel has run;  what = 1: dprobs has landed too (the step is over).       */
typedef struct zs_host_step zs_host_step;
int zs_host_step_create(zs_host_step** handle);
int zs_host_step_destroy(zs_host_step* handle);
int64_t zs_iw_step_host_workspace(int64_t K, int64_t B, int64_t X);
int zs_iw_step_host(zs_host_step* handle, int estimator, float* cost_host, float* dprobs_host, float* dlogp_host,
                    float* dlogq_host, const float* probs_host, const float* x_host, const float* logp_other_host,
                    const float* logq_host, int64_t K, int64_t B, int64_t X, double grad_scale, void* ws,
                    int64_t ws_bytes, zs_stream_t stream);
int zs_iw_step_host_begin(zs_host_step* handle, int estimator, float* cost_host, float* dprobs_host, float* dlogp,
                          float* dlogq, const float* probs_host, const float* x_host, const float* logp_other,
                          const float* logq, int64_t K, int64_t B, int64_t X, double grad_scale, void* ws,
                          int64_t ws_bytes, int scalars_on_device, zs_stream_t stream);
int zs_iw_step_host_wait(zs_host_step* handle, int what);

#ifdef __cplusplus
}
#endif
#endif /* ZS_B200_H */
