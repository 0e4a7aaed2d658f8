/*
 * mcmcn.h -- C ABI of the B200-native MCMC engine for nested data.
 *
 * This is the drop-in boundary of the hot path behind the reference's
 *   posteriorSampling.samplePosterior   (/root/reference/posteriorSampling.py:28-216)
 *   sampleDiagnosis.diagnoseSamples     (/root/reference/sampleDiagnosis.py:11-85)
 * The reference has no FFI: its boundary is those two Python signatures, kept
 * verbatim by mcmc-for-nested-data_b200/{posteriorSampling,sampleDiagnosis}.py,
 * which bind this library with ctypes (see INTEGRATION.md).  Everything here is
 * plain pointers and sizes; no torch types.  All `device` pointers are CUDA
 * device pointers owned by the caller; `stream` is a cudaStream_t (NULL = the
 * legacy default stream).  Every entry point returns MCMCN_OK (0) or a negative
 * error code; mcmcn_last_error() gives the message of the last failure on the
 * calling thread.
 *
 * Layout conventions (S = mcmcn_state.stride, the padded chain count):
 *   per-(name, group, chain) arrays are [P][G][S] with the chain index fastest,
 *   so that a warp of 32 chains reads/writes 256 contiguous bytes;
 *   per-(group, chain) arrays are [G][S]; hyper-parameters are [5][P][S].
 */
#ifndef MCMCN_H
#define MCMCN_H

#ifdef __CUDACC_RTC__
typedef int int32_t;
typedef unsigned int uint32_t;
typedef long long int64_t;
typedef unsigned long long uint64_t;
typedef unsigned char uint8_t;
#else
#include <stdint.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define MCMCN_VERSION 100
#define MCMCN_MAX_PARAMS 17          /* P <= 17 (K <= 16 regression coefficients + sigma) */

/* error codes */
#define MCMCN_OK 0
#define MCMCN_ERR_INVALID (-1)       /* bad argument / unsupported configuration */
#define MCMCN_ERR_CUDA (-2)          /* a CUDA runtime call failed */
#define MCMCN_ERR_UNSUPPORTED (-3)   /* objective / shape not compiled in and NVRTC unavailable */
#define MCMCN_ERR_NVRTC (-4)         /* user objective failed to compile */

/* objective registry: the device restatement of the reference's user callable
 * (posteriorSampling.py:61-102 contract; examples example/distribution.py:18-24,
 * example/regression.py:53-67). */
#define MCMCN_OBJ_GAUSSIAN_DISTRIBUTION 0
#define MCMCN_OBJ_LINEAR_REGRESSION 1
#define MCMCN_OBJ_BERNOULLI_LOGIT 2
#define MCMCN_OBJ_USER 3             /* NVRTC-compiled user source, see mcmcn_user_objective_* */

/* pooling (posteriorSampling.py:1040-1043, :1146-1148) */
#define MCMCN_POOL_PARTIAL 0
#define MCMCN_POOL_NONE 1
#define MCMCN_POOL_COMPLETE 2

/* prior families for none/complete pooling (scipy.stats frozen distributions
 * the reference accepts in `priorDistribution`, posteriorSampling.py:293-294) */
#define MCMCN_PRIOR_NORM 0
#define MCMCN_PRIOR_GAMMA 1
#define MCMCN_PRIOR_UNIFORM 2
#define MCMCN_PRIOR_EXPON 3
#define MCMCN_PRIOR_HALFNORM 4
#define MCMCN_PRIOR_LOGNORM 5     /* a = s */
#define MCMCN_PRIOR_CAUCHY 6
#define MCMCN_PRIOR_T 7           /* a = df */
#define MCMCN_PRIOR_BETA 8        /* a, b */
#define MCMCN_PRIOR_INVGAMMA 9    /* a */
#define MCMCN_PRIOR_LAPLACE 10
#define MCMCN_PRIOR_LOGISTIC 11
#define MCMCN_PRIOR_CHI2 12       /* a = df */

typedef struct mcmcn_prior {
    int32_t family;
    int32_t reserved;
    double a;            /* first shape parameter (gamma a, lognorm s, t / chi2 df, beta a, invgamma a) */
    double loc;
    double scale;
    double log_scale;    /* log(scale), precomputed by the host in fp64 */
    double c0;           /* family constant, precomputed by the host in fp64: gammaln(a) (gamma, invgamma),
                            2 s^2 (lognorm), log(poch(df/2, 1/2)) - (log(df) + log(pi))/2 (t), betaln(a, b) (beta),
                            gammaln(df/2) (chi2) */
    double b;            /* second shape parameter (beta b); chi2: log(2) df / 2 */
} mcmcn_prior;

/* The model: objective + observation data + group structure + priors.
 * `data` holds one packed block per group, group g at element offset
 * group_off[g] (group_off has G+1 entries; elements are float when
 * precision == 32 and double when precision == 64).  Block layouts:
 *   linear_regression   ceil(R/4) quads of [KP][4 obs] x then [4] ne, KP = K rounded up to 4;
 *                       ne = x.bbar_g - y with bbar_g the group's reference point, obj_const[g*K+k]
 *   bernoulli_logit     ceil(R/4) quads of [4] x then [4] y
 *   gaussian_distribution  ceil(R/4) quads of [4 obs][PP] mu_j of the observation's group, PP = P rounded up to 4
 * (padding observations are zero).  Tasks are runs of consecutive groups
 * [task_group0[t], task_group0[t+1]) whose blocks are staged into shared
 * memory by one TMA bulk copy. */
typedef struct mcmcn_model {
    int32_t objective;
    int32_t n_params;        /* P */
    int32_t n_coef;          /* K (linear_regression), else 0 */
    int32_t precision;       /* 32: FP32 observation math, FP64 group sums; 64: all FP64 */
    int32_t pooling;
    int32_t n_groups;        /* G as stepped (1 for complete pooling) */
    int32_t n_tasks;
    int32_t n_obj_const;
    int64_t n_obs;           /* N */
    const void* data;            /* device */
    const int64_t* group_off;    /* device [G+1] */
    const int32_t* group_nobs;   /* device [G] */
    const int32_t* task_group0;  /* device [n_tasks+1] */
    const int32_t* task_group0_host; /* host copy of the same table */
    const int64_t* group_off_host;   /* host copy [G+1] */
    const double* obj_const;     /* device objective constants (gaussian_distribution: sd[P], log sd[P];
                                    linear_regression: bbar[G][K]) */
    const void* user_objective;  /* handle from mcmcn_user_objective_compile, or NULL */
    /* Tensor-core operand blocks (linear_regression, precision 32, K <= 16; NULL = not provided, the
     * FP32-pipe kernel is used).  Block of group g at float offset tc_group_off[g]: 2 KB + 1 slabs of
     * [Np][8] floats, Np = R rounded up to 16 (at least 16), KB = 1 for K <= 8 and 2 for K = 9..16:
     * X_hi of coefficients 0-7 (then 8-15), X_lo likewise, NE, where x = x_hi + x_lo with both parts
     * rounded to TF32, and NE row n = (ne_hi, ne_mid, ne_lo, 0, 0, 0, 0, 0) with
     * ne = ne_hi + ne_mid + ne_lo exactly.  Within a slab element (n, k) sits at float index
     * (n/8)*64 + (k/4)*32 + (n%8)*4 + (k%4): the K-major, no-swizzle shared-memory layout that
     * tcgen05.mma reads (8-row x 16-byte core matrices).  Padding rows and coefficients are zero. */
    const void* tc_data;             /* device float */
    const int64_t* tc_group_off;     /* device [G+1], in floats */
    int64_t tc_max_block_floats;     /* largest block */
    mcmcn_prior prior[MCMCN_MAX_PARAMS];   /* none / complete pooling only */
    /* Complete pooling at scale (optional, NULL = step the single group of all N observations with
     * one warp per 128 chains).  `split` describes the SAME observations as many small groups (its
     * pooling field is ignored); each sweep then evaluates the proposal's log-likelihood over those
     * groups in parallel (observations x chains across the whole GPU), sums the partial sums in group
     * order per chain and takes the decision in a per-chain kernel (CompletePooling,
     * posteriorSampling.py:662-685); mcmcn_group_loglik evaluates over the same groups.  Environment
     * variable MCMCN_NO_SPLIT=1 ignores `split` in both.  `split_scratch`: device,
     * (P + split->n_groups + 3) * stride doubles, working memory of mcmcn_run and mcmcn_group_loglik. */
    const struct mcmcn_model* split;
    double* split_scratch;
} mcmcn_model;

/* Chain state of the n_chains chains resident on this device
 * (reference: Parameter / HyperParameter objects, posteriorSampling.py:234-511). */
typedef struct mcmcn_state {
    int32_t n_chains;
    int32_t stride;          /* S >= n_chains, multiple of 32 */
    int64_t chain_id0;       /* global id of local chain 0: Philox key, so results do not depend on the GPU count */
    double* theta;           /* [P][G][S] Parameter._value */
    double* scale;           /* [P][G][S] Parameter._adaptiveScaleFactor */
    uint32_t* counts;        /* [P][G][S] nAccepted | nRejected << 16 since the last tune */
    double* ll;              /* [G][S]    group log-likelihood (NaN = never set, :265) */
    double* lprior;          /* [P][G][S] Parameter._logPrior (fixed priors; partial: iteration-0 override, may be NULL) */
    double* hyper;           /* [5][P][S] mu, sigma2, sd = sqrt(sigma2), log sd, 1/sd (partial pooling) */
} mcmcn_state;

/* One call advances all chains by n_iter iterations of Sampler._loop
 * (posteriorSampling.py:862-896). */
typedef struct mcmcn_run_args {
    int64_t iter0;           /* index of the first iteration of this call */
    int32_t n_iter;
    int32_t burn;
    int32_t thin;
    int32_t tune_interval;   /* 100 in the reference (:1157) */
    uint64_t seed;           /* Philox key word 1 (word 0 is the global chain id) */
    /* replay tape, all NULL for free-running Philox; laid out per iteration of this call */
    const double* tape_z;        /* [n_iter][P][G][S] standard normal behind each proposal */
    const double* tape_u;        /* [n_iter][P][G][S] uniform of each accept test */
    const uint8_t* tape_accept;  /* [n_iter][P][G][S] decisions to force (teacher forcing), or NULL */
    const double* tape_zmu;      /* [n_iter][P][S] standard normal behind each mu draw */
    const double* tape_qsig;     /* [n_iter][P][S] unit inverse-gamma draw behind each sigma2 */
    /* per-decision trace, all NULL for none; [n_iter][P][G][S] */
    double* trace_ll;            /* proposal group log-likelihood */
    double* trace_lp;            /* proposal log-prior */
    double* trace_diff;          /* log-posterior difference */
    uint8_t* trace_accept;       /* the engine's own decision (before forcing) */
    /* retained-sample store, NULL for none: [rows][ncol][S], ncol = P*G (+2P for partial) */
    void* store;
    int32_t store_dtype;         /* 32 or 64 */
    int32_t use_lprior_override; /* partial pooling: read the current log-prior from state.lprior (iteration iter0 only) */
    int64_t store_row0;          /* row that the first retained iteration of this call goes to */
    int64_t store_rows;          /* capacity in rows */
    /* optional per-kernel timing (host pointer to 12 doubles that must outlive
     * mcmcn_timing_collect, accumulated into; NULL = off): [3..5] launches of the step / hyper /
     * write-back kernels (always counted); every 8th iteration's launches are bracketed by
     * CUDA events on `stream`, and mcmcn_timing_collect() adds their durations to [0..2] (ms)
     * and the number of timed launches to [6..8].  The call itself stays asynchronous. */
    double* timing;
    /* optional pointwise log-likelihood of every retained state (saveLogLikelihood,
     * posteriorSampling.py:890-891, :907-909): device double [store_rows][N][S], written at the same row
     * index as `store` (which must be given); NULL = off */
    double* loglik_store;
} mcmcn_run_args;

int mcmcn_version(void);
const char* mcmcn_last_error(void);

/* Number of bytes of observation data one task may stage in shared memory. */
int mcmcn_tile_capacity_bytes(void);

/* Is (objective, n_coef, n_params, precision) compiled in? 1 yes, 0 no. */
int mcmcn_supported(int objective, int n_params, int n_coef, int precision);

/* Will mcmcn_run advance this model with the tcgen05 step kernel (1) or the FP32-pipe kernel (0)?
 * (linear_regression, precision 32, K <= 16, tc_data given, every group block within the stage
 * capacity; environment variable MCMCN_NO_TC=1 forces 0.) */
int mcmcn_uses_tensor_core(const mcmcn_model* model);

/* Replaces Sampler._loop + StepMethod.step (posteriorSampling.py:594-613, :862-896). */
int mcmcn_run(const mcmcn_model* model, const mcmcn_state* state,
              const mcmcn_run_args* args, void* stream);

/* Wait for and read back the events recorded by mcmcn_run calls of this thread that had
 * `timing` set (see mcmcn_run_args.timing). */
int mcmcn_timing_collect(void);

/* Group log-likelihood of the current state (posteriorSampling.py:629-635 with
 * proposedParameter=None).  out_ll is device [G][S].  If pooled_theta (device
 * [P][S]) is not NULL every group uses those values instead of state.theta
 * (MCMC._mleObjectiveFunction, :1102-1105).  With a split model (complete pooling at scale,
 * mcmcn_model.split) the log-likelihood is evaluated per small group into split_scratch and
 * out_ll[0][c] is their sum, from 0.0 in group order, for every chain c < n_chains; lanes
 * from n_chains on are unspecified. */
int mcmcn_group_loglik(const mcmcn_model* model, const mcmcn_state* state,
                       const double* pooled_theta, double* out_ll, void* stream);

/* out[c] = -sum_g ll[g][c] in group order (:1105). ll device [G][S], out device [S]. */
int mcmcn_pooled_nll(int n_groups, int stride, const double* ll, double* out, void* stream);

/* Pointwise log-likelihood of the current state (StepMethod.logLikelihood,
 * posteriorSampling.py:656-659).  out is device [N][S] double. */
int mcmcn_pointwise_loglik(const mcmcn_model* model, const mcmcn_state* state,
                           double* out, void* stream);

/* ---- diagnostics (sampleDiagnosis.py:158-255, :419-427, :766-776) ----------
 * x is device double [n_keys][m][n]: key-major, then half-chain, then draw. */
/* Half-chains of n_keys columns [k0, k0 + n_keys) of a sample store (device [rows][ncol][stride], chain
 * fastest, store_dtype 32 or 64; rows 0 .. 2n-1 are used) into out, device double [n_keys][out_m][n]:
 * half-chain out_j0 + 2c + h = rows h n .. h n + n - 1 of chain c < n_chains (sampleDiagnosis.py:118-156).
 * Several stores (shards of the chains) fill one `out` through out_j0. */
int mcmcn_diag_halfchains(const void* store, int32_t store_dtype, int32_t n, int64_t ncol, int64_t stride,
                          int64_t k0, int64_t n_keys, int32_t n_chains, int32_t out_m, int32_t out_j0,
                          double* out, void* stream);
/* per half-chain mean and ddof=1 variance: out_mean, out_var device [n_keys][m] */
int mcmcn_diag_moments(const double* x, int64_t n_keys, int32_t m, int32_t n,
                       double* out_mean, double* out_var, void* stream);
/* per-lag sum over half-chains of squared differences: out device [n_keys][n],
 * out[k][t] = sum_j sum_{i>=t} (x[k][j][i]-x[k][j][i-t])^2  (numerator of :189-194) */
int mcmcn_diag_variogram(const double* x, int64_t n_keys, int32_t m, int32_t n,
                         double* out, void* stream);
/* B, W, vhat, rhat per key from the half-chain moments (:158-187, :216-224): out device [n_keys][4] */
int mcmcn_diag_rhat(const double* mean, const double* var, int64_t n_keys, int32_t m, int32_t n,
                    double* out, void* stream);
/* autocorrelation, truncation and effective sample size per key (:196-208, :232-255) from the
 * variogram numerators and the [n_keys][4] output of mcmcn_diag_rhat; rho_out (device
 * [n_keys][n]) may be NULL; ess_out is device [n_keys]. m is the TOTAL number of half-chains. */
int mcmcn_diag_ess(const double* vario, const double* rhat4, int64_t n_keys, int32_t m, int32_t n,
                   double* rho_out, double* ess_out, void* stream);
/* mean of each contiguous row of `len` doubles (Summary's mean over groups, :466-470) */
int mcmcn_diag_row_mean(const double* x, int64_t rows, int64_t len, double* out, void* stream);
/* in-place ascending sort of each key's m*n pooled draws (for median / HDI, :419-427) */
int mcmcn_diag_sort_keys(double* x, int64_t n_keys, int64_t len, void* stream);
/* numpy.median and computeHpdInterval (:766-776) on sorted keys: out device [n_keys][3] =
 * median, HDI lower, HDI upper; gap = max(1, min(len-1, round(len*p))) is computed by the
 * caller (Python banker's rounding); first minimum-width interval wins. */
int mcmcn_diag_median_hdi(const double* sorted, int64_t n_keys, int64_t len, int64_t gap,
                          double* out, void* stream);

/* ---- measured pipe peaks for the roofline (SURVEY.md section 8d) -----------
 * Run an FFMA-only / MUFU-only / MMA-only microbenchmark on the current device and return
 * the achieved rate in *out (FP32 flop/s, MUFU op/s, TF32 flop/s). */
int mcmcn_peak_fp32(double* out_flops, void* stream);
int mcmcn_peak_mufu(double* out_ops, void* stream);
/* tensor pipe: back-to-back tcgen05.mma kind::tf32 of the step kernel's shape (M 128, N 208, K 8), FLOP/s */
int mcmcn_peak_tf32(double* out_flops, void* stream);

/* ---- user objectives (north star (1): documented C ABI, compiled by NVRTC) ----
 * `source` is CUDA C++ that defines, at namespace scope,
 *
 *   __device__ mcmc_real mcmc_obj_loglik(const mcmc_real* theta,  // P values of this observation's group
 *                                        const mcmc_real* obs,    // this observation's record (obs_floats values)
 *                                        const mcmc_real* hdr,    // the group's header (hdr_floats values)
 *                                        int obs_index,           // index within the group
 *                                        int group);
 *
 * returning the pointwise log-likelihood (NaN / -inf are meaningful: they reject,
 * posteriorSampling.py:354-360).  `mcmc_real` is float (precision 32) or double (64).
 * The contract is the reference's (posteriorSampling.py:61-102): ll may depend only on
 * the observation's own record and its own group's parameters.  Records are laid out
 * group-contiguously: block g = [hdr_floats header][R_g * obs_floats records], both
 * multiples of 4 values.  A plain host callable cannot be used; there is no CPU path. */
int mcmcn_user_objective_compile(const char* source, int32_t n_params, int32_t obs_floats,
                                 int32_t hdr_floats, int32_t precision, void** out_handle);
int mcmcn_user_objective_free(void* handle);

/* ---- the chains' host random streams of the start state (host memory, no device work) ----
 * The reference runs each chain in its own process and seeds numpy's global legacy generator with the chain
 * index (posteriorSampling.py:225, :1015); the start state is drawn from that stream: numpy.random.uniform per
 * parameter (:1069-1077) and, under partial pooling, numpy.random.normal per parameter and group (:738-758).
 * Stream i of a handle is numpy.random.RandomState(seed0 + i): MT19937 seeded by init_genrand, 53-bit doubles,
 * the polar normal with its cached second value -- bit for bit.  `threads` host threads share the listed streams.
 *   uniform: for every listed stream j, `count` draws low[i] + (high[i] - low[i]) * u_i  -> out[j][i]
 *   normal:  for every listed stream j, out[out_off[j] .. out_off[j+1]) standard normals, in order
 *   get/set_state: numpy's ('MT19937', key[624], pos, has_gauss, cached_gaussian) tuple of one stream, to hand
 *            a stream to scipy (`prior.rvs(random_state=...)`, :1079-1081) and take it back. */
int mcmcn_streams_create(int64_t n, int64_t seed0, int32_t threads, void** out_handle);
int mcmcn_streams_free(void* handle);
int mcmcn_streams_uniform(void* handle, const int64_t* which, int64_t n_which, int32_t count, const double* low,
                          const double* high, double* out, int32_t threads);
int mcmcn_streams_normal(void* handle, const int64_t* which, int64_t n_which, const int64_t* out_off, double* out,
                         int32_t threads);
int mcmcn_streams_get_state(void* handle, int64_t i, uint32_t* key624, int32_t* pos, int32_t* has_gauss, double* gauss);
int mcmcn_streams_set_state(void* handle, int64_t i, const uint32_t* key624, int32_t pos, int32_t has_gauss, double gauss);

/* Known-answer hook for tests: out[0..3] = Philox4x32-10(counter[0..3], key[0..1]) computed on
 * the device (all three are device pointers to uint32). */
int mcmcn_debug_philox(const void* counter, const void* key, void* out);

/* Distribution-test hook: n draws of one of the step path's own samplers, one Philox key per draw
 * (key = draw index, `seed`), written to the device array `out`:
 *   SWEEP_NORMALS   out[2n]: both Box-Muller branches behind two consecutive sweeps' proposals
 *   SWEEP_UNIFORMS  out[2n]: the two accept-test uniforms of the same Philox call
 *   HYPER_NORMAL    out[n]:  the standard normal behind the Gibbs mu draw (posteriorSampling.py:485-487)
 *   UNIT_INVGAMMA   out[n]:  1 / Gamma(a, 1) (Marsaglia-Tsang), the unit-scale draw behind sigma2
 *                            (posteriorSampling.py:489-498: scipy.stats.invgamma(a).rvs())
 *   UNIFORM53       out[n]:  the 53-bit uniform of the gamma sampler's accept test */
#define MCMCN_DRAW_SWEEP_NORMALS 0
#define MCMCN_DRAW_SWEEP_UNIFORMS 1
#define MCMCN_DRAW_HYPER_NORMAL 2
#define MCMCN_DRAW_UNIT_INVGAMMA 3
#define MCMCN_DRAW_UNIFORM53 4
int mcmcn_debug_draws(int kind, int64_t n, uint64_t seed, double a, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MCMCN_H */
