/*
 * extmcmc.h -- C ABI of libextmcmc_cuda.so
 *
 * B200-native (sm_100a) engine for the one data-parallel hot path of
 * ExtensibleMCMC.jl: the Metropolis-Hastings transition step
 * (proposal -> log-likelihood + log-prior -> accept/reject -> adaptation ->
 * chain statistics) executed for many independent chains against one shared
 * observation set.
 *
 * This header is the drop-in boundary.  A Julia `CUDAMCMCBackend <: MCMCBackend`
 * (reference seam: src/types.jl:107-117, src/mcmc.jl:39-48) binds these symbols
 * with `ccall((:extmcmc_xxx, "libextmcmc_cuda"), ...)`; in this repository the
 * Python host mirror binds them through ctypes.  See INTEGRATION.md.
 *
 * Conventions
 *  - plain C: POD structs, raw pointers, sizes; no C++/torch types; no exceptions
 *    cross the boundary; every function returns an int32 status (0 = OK).
 *  - all real numbers are IEEE binary64 (the reference computes in Float64).
 *  - chain-major SoA: a per-chain quantity q with K components is laid out
 *    q[k * n_chains + c] ("chain fastest").
 *  - coordinates and update indices are 0-based here (the Julia shim subtracts 1).
 *  - host buffers are caller-owned; the library copies in / fills out and never
 *    retains a host pointer after the call returns.
 *  - a handle is not thread-safe.
 */
#ifndef EXTMCMC_H_
#define EXTMCMC_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EXTMCMC_ABI_VERSION 2

/* ---- status codes -------------------------------------------------------- */
enum {
    EXTMCMC_OK           = 0,
    EXTMCMC_EINVAL       = -1, /* bad argument / call order                    */
    EXTMCMC_EUNSUPPORTED = -2, /* law / prior / kernel not implemented on GPU;
                                  mirrors the reference's error("... not
                                  implemented") convention, src/updates.jl:42-53 */
    EXTMCMC_ECUDA        = -3, /* CUDA runtime error                           */
    EXTMCMC_ENCCL        = -4, /* NCCL error                                   */
    EXTMCMC_EOOM         = -5, /* device or host allocation failed             */
    EXTMCMC_EDOMAIN      = -6, /* a chain reached law parameters outside the
                                  law's domain (the reference throws there,
                                  e.g. PosDefException in MvNormal(mu, Sigma),
                                  src/example/gsn_target.jl:20)                */
    EXTMCMC_ESTALE       = -7  /* history rows requested were overwritten      */
};

/* ---- target laws (reference: user law with set_parameters!/loglikelihood,
 *      docs/src/get_started/basic_use.md; shipped: src/example/gsn_target.jl) */
enum {
    EXTMCMC_LAW_GSN_IID_1D  = 1, /* GsnTargetLaw, d = 1: theta = [mu, sigma^2]  */
    EXTMCMC_LAW_GSN_MV      = 2, /* GsnTargetLaw, general d: theta = [mu; vec(Sigma)]
                                    (src/example/gsn_target.jl:1-29)            */
    EXTMCMC_LAW_LOGISTIC    = 3, /* Bayesian logistic regression, theta = beta[d]
                                    (no reference law; build-defined, cfg 3)    */
    EXTMCMC_LAW_HIER_NORMAL = 4, /* hierarchical normal, theta = [theta_1..G, mu, tau]
                                    (no reference law; build-defined, cfg 4)    */
    EXTMCMC_LAW_USER        = 5  /* user-defined law: CUDA C++ source compiled at run time,
                                    see extmcmc_set_user_law                    */
};

/* ---- how a user-defined law provides its gradient (with_grad of extmcmc_set_user_law) */
enum {
    EXTMCMC_USER_GRAD_NONE    = 0, /* no gradient: no MALA, no extmcmc_eval_grad            */
    EXTMCMC_USER_GRAD_HAND    = 1, /* the source defines logpdf_grad (any other non-zero
                                      value than EXTMCMC_USER_GRAD_FORWARD means the same)   */
    EXTMCMC_USER_GRAD_FORWARD = 2  /* the source is generic over its scalar; the library
                                      derives the gradient in forward mode (dual numbers)    */
};
/* ---- what a user-defined law declares besides logpdf (flags of extmcmc_set_user_law_ex) */
enum {
    EXTMCMC_USER_THETA_TERM = 1    /* the source defines logpdf_theta (+ logpdf_theta_grad with a
                                      hand-written gradient): a term of theta only, added once */
};

/* ---- transition kernels (src/transition_kernels/random_walk.jl, src/updates.jl) */
enum {
    EXTMCMC_KERNEL_RW_UNIFORM   = 1, /* UniformRandomWalk, random_walk.jl:45-94  */
    EXTMCMC_KERNEL_RW_GAUSS     = 2, /* GaussianRandomWalk, :123-171             */
    EXTMCMC_KERNEL_RW_GAUSS_MIX = 3, /* GaussianRandomWalkMix, :193-232          */
    EXTMCMC_KERNEL_MALA         = 4  /* MALAUpdate (stub in reference, updates.jl:216-218):
                                        th° = th + tau^2/2 grad(ll + log prior)(th) + tau z;
                                        step = tau[1]; priors: IMPROPER, NORMAL            */
};

/* ---- priors (src/priors.jl) ---------------------------------------------- */
enum {
    EXTMCMC_PRIOR_IMPROPER     = 0, /* ImproperPrior: 0.0             priors.jl:18-19 */
    EXTMCMC_PRIOR_IMPROPER_POS = 1, /* ImproperPosPrior: -sum(log th)  priors.jl:25-26 */
    EXTMCMC_PRIOR_NORMAL       = 2, /* StandardPrior(Normal(m, s)) on each coordinate
                                       (iid product), params = {m, s}  priors.jl:35-39 */
    EXTMCMC_PRIOR_GAMMA        = 3, /* StandardPrior(Gamma(shape, scale)) iid product,
                                       params = {shape, scale}; -Inf for th <= 0      */
    EXTMCMC_PRIOR_UNIFORM      = 4, /* StandardPrior(Uniform(a, b)) iid product,
                                       params = {a, b}; -Inf outside [a, b]           */
    EXTMCMC_PRIOR_PRODUCT      = 5, /* ProductPrior(dists, dims), priors.jl:60-88: factors over
                                       consecutive coordinate groups; params = {K, then per
                                       factor: kind (any iid family), dim, p0, p1}, K <= 16   */
    /* further StandardPrior families (iid product over the update's coordinates; the closed
       forms of Distributions.jl's logpdf, -Inf outside the support)                           */
    EXTMCMC_PRIOR_EXPONENTIAL  = 6, /* Exponential(scale): params = {scale}                    */
    EXTMCMC_PRIOR_INV_GAMMA    = 7, /* InverseGamma(shape, scale)                              */
    EXTMCMC_PRIOR_BETA         = 8, /* Beta(alpha, beta)                                       */
    EXTMCMC_PRIOR_LOGNORMAL    = 9, /* LogNormal(mu, sigma)                                    */
    EXTMCMC_PRIOR_CAUCHY       = 10, /* Cauchy(mu, sigma)                                      */
    EXTMCMC_PRIOR_MVNORMAL     = 11, /* StandardPrior(MvNormal(mu, Sigma)) on the whole coordinate
                                        block of a joint update (priors.jl:35-39 wraps any
                                        Distributions object): params = {mu[p_u], L[p_u*p_u]}, L the
                                        lower Cholesky factor of Sigma, column-major (the host side
                                        factorises; the device whitens, as PDMats does)            */
    EXTMCMC_PRIOR_USER         = 12  /* user-defined prior: CUDA C++ logprior compiled at run time
                                        (extmcmc_set_user_prior); params = its pp[]               */
};

/* ---- adaptation schemes (src/transition_kernels/adaptation.jl) ----------- */
enum {
    EXTMCMC_ADAPT_NONE    = 0, /* NoAdaptation, adaptation.jl:26                  */
    EXTMCMC_ADAPT_UNIF_RW = 1, /* AdaptationUnifRW, adaptation.jl:51-71,273-329   */
    EXTMCMC_ADAPT_HAARIO  = 2, /* HaarioTypeAdaptation, adaptation.jl:372-426     */
    EXTMCMC_ADAPT_MALA    = 3  /* acceptance-rate targeting of the MALA step tau with
                                  the same +-delta rule as AdaptationUnifRW        */
};

/* ---- how work is split when several ranks (one process per GPU) cooperate  */
enum {
    EXTMCMC_SHARD_CHAINS = 0, /* each rank owns a disjoint chain range, observations
                                 replicated, no communication                      */
    EXTMCMC_SHARD_OBS    = 1  /* each rank owns a slice of the observations, chain
                                 state replicated, per-chain partial log-likelihoods
                                 all-reduced (NCCL) once per update step           */
};

/* ---- randomness source ---------------------------------------------------- */
enum {
    EXTMCMC_RNG_PHILOX = 0, /* per-chain Philox4x32-10 counter stream               */
    EXTMCMC_RNG_REPLAY = 1  /* proposals and Exp(1) draws supplied by the caller    */
};

/* Parameters of AdaptationUnifRW (adaptation.jl:51-61); scalars only -- the
 * reference's run path works only for scalar scale/min/max/offset
 * (compute_delta does max(1.0, vector), adaptation.jl:312-319). */
typedef struct extmcmc_adapt {
    int32_t kind;                 /* EXTMCMC_ADAPT_*                               */
    int32_t adapt_every_k_steps;  /* default 100                                   */
    double  target_accpt_rate;    /* default 0.234                                 */
    double  scale;                /* default 1.0                                   */
    double  min;                  /* default 1e-12                                 */
    double  max;                  /* default 1e7                                   */
    double  offset;               /* default 1e2                                   */
} extmcmc_adapt_t;

/* One update = transition kernel + coordinate subset + prior + adaptation
 * (RandomWalkUpdate, src/updates.jl:163-183). */
typedef struct extmcmc_update {
    int32_t        kernel;        /* EXTMCMC_KERNEL_*                              */
    int32_t        n_coords;      /* p_u = length(coords)                          */
    const int32_t *coords;        /* [p_u] 0-based indices into theta              */
    const double  *step;          /* RW_UNIFORM: eps[p_u] (UniformRandomWalk.eps);
                                     RW_GAUSS: Sigma[p_u*p_u] column-major;
                                     RW_GAUSS_MIX: Sigma_A, Sigma_B, lambda
                                     (2*p_u*p_u + 1); MALA: tau[1].
                                     p_u <= 32 for the random walks, any p_u for MALA */
    const uint8_t *pos;           /* [p_u] 1 = coordinate restricted to be positive */
    int32_t        prior;         /* EXTMCMC_PRIOR_*                               */
    int32_t        n_prior_params;
    const double  *prior_params;
    extmcmc_adapt_t adapt;
} extmcmc_update_t;

/* One element of the MCMCSchedule iterator (src/schedule.jl:56-66):
 * (prev_mcmciter, prev_pidx, mcmciter, pidx).  mcmciter is 1-based as in the
 * reference (it enters the adaptation rule, adaptation.jl:312-319); pidx is
 * 0-based; prev_pidx = -1 encodes `nothing` (first step). */
typedef struct extmcmc_step {
    int64_t mcmciter;
    int64_t prev_mcmciter;
    int32_t pidx;
    int32_t prev_pidx;
} extmcmc_step_t;

typedef struct extmcmc_config {
    int32_t  abi_version;     /* EXTMCMC_ABI_VERSION                               */
    int32_t  device;          /* CUDA device ordinal                               */
    int64_t  n_chains;        /* chains resident on this rank                      */
    int64_t  chain_offset;    /* global id of local chain 0 (Philox key space is
                                 global, so results do not depend on the sharding) */
    int32_t  n_params;        /* p = length(theta)                                 */
    int32_t  n_updates;       /* NU                                                */
    int32_t  law;             /* EXTMCMC_LAW_*                                     */
    int32_t  obs_dim;         /* d (1 for GSN_IID_1D)                              */
    uint64_t seed;            /* Philox key                                        */
    int32_t  shard_mode;      /* EXTMCMC_SHARD_*                                   */
    int32_t  rank;            /* this process' rank  (0 if single)                 */
    int32_t  world_size;      /* number of ranks     (1 if single)                 */
    int32_t  history_window;  /* device history ring length in update steps (>= 1) */
    int32_t  roll_window;     /* GenericChainStats.roll_window, default 100
                                 (src/chain_statistics.jl:27)                      */
    int32_t  use_graphs;      /* 1: run_block replays a captured CUDA graph        */
    int32_t  instrument;      /* 1: bracket every likelihood sweep launch with
                                 CUDA events (see extmcmc_get_sweep_time)          */
    int32_t  sweep_variant;   /* 0 = auto; 1 = "chains" mapping, 2 = "obs" mapping;
                                 11/12/14/18 = "chains" with 1/2/4/8 chains per thread */
    int32_t  stats_mode;      /* 0 = running mean + full covariance per chain (the
                                 reference's GenericChainStats); 1 = mean + diagonal
                                 of the covariance only; 2 = no running moments     */
    int32_t  reserved_[3];
} extmcmc_config_t;

typedef struct extmcmc_handle *extmcmc_t;

/* ---- lifecycle ------------------------------------------------------------ */
/* Replaces init_global_workspace(::MCMCBackend, ...) src/workspaces.jl:38-47,215-234
 * and create_workspace(...) src/workspaces.jl:280-287,460-473: allocates the
 * device-resident chain state (theta, theta_prop, ll, eps, counters, moments). */
int32_t extmcmc_create(const extmcmc_config_t *cfg, extmcmc_t *out);
int32_t extmcmc_destroy(extmcmc_t h);
/* Library-owned string, valid until the next call on the same handle
 * (h == NULL: last error of a failed extmcmc_create). */
const char *extmcmc_last_error(extmcmc_t h);
int32_t extmcmc_abi_version(void);

/* ---- model, data, updates ------------------------------------------------- */
/* Replaces the user's law object + its observations: data = (P = law, obs = ...)
 * (src/workspaces.jl:229-237).  Row-major obs[n_obs][obs_dim]; y = responses (LOGISTIC)
 * or the 0-based group index of every observation, sorted ascending (HIER_NORMAL);
 * NULL otherwise.  The library copies.  n_obs >= 1 (EXTMCMC_EINVAL otherwise).
 * (EXTMCMC_LAW_USER: rows of obs_dim columns, y = NULL.)
 * Under EXTMCMC_SHARD_OBS each rank uploads only its own slice. */
int32_t extmcmc_upload_obs(extmcmc_t h, const double *obs, int64_t n_obs,
                           int32_t obs_dim, const double *y);
/* Observations generated on the device from Philox(seed): x ~ N(mean, sd^2),
 * global indices [first, first + n_obs) (BASELINE cfg 5: N = 1e9). */
int32_t extmcmc_generate_obs_normal(extmcmc_t h, int64_t first, int64_t n_obs,
                                    double mean, double sd, uint64_t seed);
/* ---- user-defined laws (EXTMCMC_LAW_USER) ----------------------------------
 * The reference's user law -- set_parameters!(P, theta) and loglikelihood(P, obs) -- written as one
 * string of CUDA C++ (not Julia) that defines:
 *
 *   struct Law { ... };   per-chain constants, kept in registers for the whole sweep
 *   // set_parameters!(P, theta): th[0..P-1] = the chain's full parameter vector; return false when
 *   // theta is outside the law's domain (the chain's ll is then NaN, its proposal is rejected and
 *   // extmcmc_sync returns EXTMCMC_EDOMAIN)
 *   __device__ bool set_parameters(Law &L, const double *th);
 *   // one term of loglikelihood(P, obs): x[0..D-1] = one observation row
 *   __device__ double logpdf(const Law &L, const double *x);
 *   // optional (with_grad = 1; needed by MALA and extmcmc_eval_grad): returns logpdf and ADDS
 *   // d logpdf / d th into g[0..P-1]
 *   __device__ double logpdf_grad(const Law &L, const double *x, double *g);
 *
 * Forward mode (with_grad = EXTMCMC_USER_GRAD_FORWARD): the same law written once, generic over its
 * scalar, and no logpdf_grad -- the gradient is derived as ForwardDiff derives it from generic Julia:
 *
 *   template <class real> struct Law { ... };   every parameter-dependent field of type real
 *   template <class real> __device__ bool set_parameters(Law<real> &L, const real *th);
 *   template <class real> __device__ real logpdf(const Law<real> &L, const double *x);   // x: data
 *
 * Value sweeps run Law<double>; gradient sweeps run Law<extmcmc::Dual<P>>, a value and its P partial
 * derivatives (csrc/dual.cuh), whose value parts are the very double operations of Law<double>: under
 * -fmad=false the log-likelihood of a gradient sweep is bit-identical to the value sweep's.  Dual
 * supports + - * / (with double operands on either side), compound assignment, comparisons (on the
 * value), exp expm1 log log1p sqrt pow fabs fmin fmax fma sin cos tanh erf erfc normcdf, isinf isnan
 * isfinite.  Any other function of a real (lgamma, ...) and any conversion of a real to double do not
 * compile (EXTMCMC_EINVAL, the log names the call).  Limit: 1 <= n_params <= 16 (each real field holds
 * n_params + 1 doubles in registers); larger is EXTMCMC_EUNSUPPORTED.
 *
 * Chunked forward mode (extmcmc_set_user_law_chunked): the same source, up to n_params = 64.  A
 * gradient is ceil(P / K) sweeps of Law<extmcmc::Dual<K>>, each seeded with the unit vectors of K
 * coordinates, as ForwardDiff's chunk mode does; the chunk width K is part of the compiled program.
 * At K = P the program, its hash and its results are those of with_grad = EXTMCMC_USER_GRAD_FORWARD;
 * with the same sweep plan every K gives the same bits.
 *
 * A term of theta only (flags = EXTMCMC_USER_THETA_TERM, extmcmc_set_user_law_ex): the reference's
 * loglikelihood may add terms that depend on theta alone, such as the hierarchical p(theta_g | mu, tau)
 * of a multilevel model, which its priors cannot express (they see only their own update's
 * coordinates).  The law then also defines, evaluated once per chain and log-likelihood evaluation on
 * the Law that set_parameters built:
 *
 *   __device__ double logpdf_theta(const Law &L);
 *   // with_grad = 1: returns logpdf_theta and ADDS d logpdf_theta / d th into g[0..P-1]
 *   __device__ double logpdf_theta_grad(const Law &L, double *g);
 *   // forward mode: generic over the scalar, differentiated like logpdf
 *   template <class real> __device__ real logpdf_theta(const Law<real> &L);
 *
 * and its log-likelihood is sum_rows logpdf(L, x) + logpdf_theta(L).  The sweep's segment 0 adds the
 * term after its own rows (ll_part[0] = fl(rows + logpdf_theta), the same for every gradient
 * component), so forward mode still gives the value sweep's ll bit for bit and every chunk width the
 * same bits.  A NaN term gives the chain ll = NaN (its proposal is rejected), as a NaN logpdf does.
 * The flag is declared, not detected: with it, a source without these functions does not compile
 * (EXTMCMC_EINVAL, the log names the function); without it, the program is the one compiled before
 * the flag existed.  The flag is part of the compiled program and of a checkpoint's law hash.
 *
 * P = n_params and D = obs_dim are the macros EXTMCMC_P / EXTMCMC_D (compile-time constants).  The
 * fixed-width integer types are defined; no header can be included.  Responses and covariates are
 * extra columns of the observation row (extmcmc_upload_obs with y = NULL).  The law is compiled for
 * sm_100a with -fmad=false: a law written like the reference rounds like it; write fma() where
 * fusion is wanted.  Limits: 1 <= n_params <= 64, 1 <= obs_dim <= 64 (registers).  Not with
 * EXTMCMC_SHARD_OBS over several ranks (EXTMCMC_EUNSUPPORTED).  Compilation needs NVRTC 12
 * (libnvrtc.so.12, loaded on first use; every built-in law runs without it). */
/* Compiles the law for the handle (law EXTMCMC_LAW_USER) and replaces the one it had; any time after
 * extmcmc_create.  Invalidates the plan and the cached graphs as extmcmc_upload_obs does.
 * EXTMCMC_EINVAL when it does not compile (extmcmc_last_error carries the NVRTC log),
 * EXTMCMC_EUNSUPPORTED when NVRTC cannot be loaded, or for a forward-mode law with n_params > 16.
 * with_grad: EXTMCMC_USER_GRAD_*.  A run or eval on an EXTMCMC_LAW_USER handle without a law returns
 * EXTMCMC_EINVAL. */
int32_t extmcmc_set_user_law(extmcmc_t h, const char *source, int32_t with_grad);
/* Compiles every kernel the library can pick for (n_params, obs_dim, with_grad) for sm_100a, without a
 * handle or a device: a law that passes cannot fail to compile later (the result is cached for the
 * process).  log (may be NULL) receives the NUL-terminated NVRTC and ptxas log (registers, spill
 * bytes), truncated to log_bytes.  Returns EXTMCMC_OK, EXTMCMC_EINVAL or EXTMCMC_EUNSUPPORTED (the log
 * then says why). */
int32_t extmcmc_user_law_check(const char *source, int32_t n_params, int32_t obs_dim, int32_t with_grad,
                               char *log, int64_t log_bytes);
/* Chunked forward mode: extmcmc_user_law_check with with_grad = EXTMCMC_USER_GRAD_FORWARD for a chunk
 * width.  chunk: a width in 1..min(16, n_params) that splits n_params into at most 16 chunks, or 0 for
 * the library's choice (n_params <= 16: the width n_params, the unchunked program; above, the balanced
 * width ceil(P / ceil(P / 5))).  chunk_used (may be NULL) receives the width compiled.  EXTMCMC_EINVAL
 * for a bad width (the log says why) or a source that does not compile, EXTMCMC_EUNSUPPORTED outside
 * 1 <= n_params <= 64 or without NVRTC. */
int32_t extmcmc_user_law_check_chunked(const char *source, int32_t n_params, int32_t obs_dim, int32_t chunk,
                                       int32_t *chunk_used, char *log, int64_t log_bytes);
/* extmcmc_set_user_law for a forward-mode law at a chunk width (chunk: as extmcmc_user_law_check_chunked).
 * A checkpoint records the width with the law: a blob written at another width is refused
 * (EXTMCMC_EINVAL), since the width can change the sweep plan and so the last bits of the sums. */
int32_t extmcmc_set_user_law_chunked(extmcmc_t h, const char *source, int32_t chunk);
/* The general form of the checks above: with_grad (EXTMCMC_USER_GRAD_*), chunk (as in
 * extmcmc_user_law_check_chunked; must be 0 unless with_grad = EXTMCMC_USER_GRAD_FORWARD) and flags
 * (EXTMCMC_USER_*; other bits are EXTMCMC_EINVAL).  chunk_used (may be NULL) receives the chunk width
 * compiled in forward mode and 0 otherwise, once the arguments are accepted. */
int32_t extmcmc_user_law_check_ex(const char *source, int32_t n_params, int32_t obs_dim, int32_t with_grad,
                                  int32_t chunk, int32_t flags, int32_t *chunk_used, char *log, int64_t log_bytes);
/* extmcmc_set_user_law with the arguments of extmcmc_user_law_check_ex.  A checkpoint written by a law
 * compiled with other flags is refused (EXTMCMC_EINVAL). */
int32_t extmcmc_set_user_law_ex(extmcmc_t h, const char *source, int32_t with_grad, int32_t chunk, int32_t flags);
/* Parameter-only coordinates (theta_only; bit k = 0-based coordinate k): coordinates that logpdf (and
 * logpdf_grad) does not depend on -- the value and gradient of every row depend only on the other
 * coordinates.  Only logpdf_theta may read them; set_parameters may read every coordinate.  Such a law
 * is compiled as a program variant (EXTMCMC_THETA_ONLY = the mask, part of the NVRTC input and of the
 * law hash): its sweeps sum rows only, and a per-chain kernel adds logpdf_theta to the row sums.  The
 * handle then keeps the row sums R and their gradient of the current state, so that a random-walk update
 * that moves only parameter-only coordinates (the mu and tau of a hierarchical model, a prior precision)
 * runs without a likelihood sweep, and a MALA update after it finds the rows' part of its current
 * gradient still valid.  EXTMCMC_DATA_CACHE=0 (read per plan) turns this cache off: every element then
 * sweeps, with the same program and kernels, and gives the same bits, log-likelihoods included.
 * The list is declared, not detected, and not verified: a false declaration gives wrong sums.  The
 * check is to run the same seed with EXTMCMC_DATA_CACHE=0 and compare: a true declaration gives
 * bit-identical histories (with logpdf_grad, when it returns the value logpdf returns, bit for bit).
 * Against the same source without the declaration, the term is added to the finished row sums instead
 * of to segment 0: ll and gradient agree to rounding (one addition associated differently).
 * flags must contain EXTMCMC_USER_THETA_TERM; theta_only must be non-zero and name coordinates below
 * n_params; otherwise EXTMCMC_EINVAL, with a message and without compiling.  The other arguments are
 * those of extmcmc_user_law_check_ex.  A checkpoint is refused across different declarations, and
 * between a declared and an undeclared law. */
int32_t extmcmc_user_law_check_theta_only(const char *source, int32_t n_params, int32_t obs_dim, int32_t with_grad,
                                          int32_t chunk, int32_t flags, uint64_t theta_only, int32_t *chunk_used,
                                          char *log, int64_t log_bytes);
int32_t extmcmc_set_user_law_theta_only(extmcmc_t h, const char *source, int32_t with_grad, int32_t chunk, int32_t flags,
                                        uint64_t theta_only);

/* ---- user-defined priors (EXTMCMC_PRIOR_USER) -------------------------------
 * The reference's open Prior type (a user subtype with logpdf(prior, th), priors.jl:4-39) as a string of
 * CUDA C++ over the update's own p_u coordinates (the compile-time macro EXTMCMC_PU); pp points to the
 * update's prior_params, so new hyperparameters need no recompilation:
 *
 *   __device__ double logprior(const double *th, const double *pp);   // -INFINITY outside the support
 *   // optional (with_grad = 1): returns logprior and ADDS d logprior / d th into g[0..PU-1]
 *   __device__ double logprior_grad(const double *th, const double *pp, double *g);
 *   // forward mode (with_grad = EXTMCMC_USER_GRAD_FORWARD), differentiated on extmcmc::Dual<PU>:
 *   template <class real> __device__ real logprior(const real *th, const double *pp);
 *
 * The rules are those of a user law: -fmad=false, no headers, the EXTMCMC_USER_GRAD_* values.  A
 * random-walk update draws its proposal inside the prior's own kernel, which redraws while logprior is
 * exactly -INFINITY (at most 60000 uniforms, as the built-in priors); a MALA update evaluates logprior and
 * its gradient at the current state and at the proposal, and needs with_grad != 0.  Limits:
 * 1 <= p_u <= 64 (p_u <= 32 for the random walks), p_u <= 16 in forward mode; beyond them
 * EXTMCMC_EUNSUPPORTED.  Not with EXTMCMC_SHARD_OBS over several ranks, nor with the persistent block
 * kernels (sweep_variant 3 / 4): EXTMCMC_EUNSUPPORTED. */
/* Compiles every kernel of the prior for (p_u, with_grad) for sm_100a, without a handle or a device;
 * log as in extmcmc_user_law_check.  EXTMCMC_OK, EXTMCMC_EINVAL (does not compile) or
 * EXTMCMC_EUNSUPPORTED (limits, no NVRTC). */
int32_t extmcmc_user_prior_check(const char *source, int32_t p_u, int32_t with_grad, char *log, int64_t log_bytes);
/* Compiles (cached by the exact input) and installs the prior of update u, which extmcmc_set_update set
 * with prior EXTMCMC_PRIOR_USER; replaces the one it had and invalidates the cached graphs.  A run on a
 * handle with such an update and no prior installed returns EXTMCMC_EINVAL; a MALA update with a prior
 * without gradient, EXTMCMC_EUNSUPPORTED. */
int32_t extmcmc_set_user_prior(extmcmc_t h, int32_t u, const char *source, int32_t with_grad);
/* logprior of update u's user prior and its gradient at the current state: lp_out[n_chains],
 * grad_out[p_u * n_chains] (d/dth_i of the update's coordinate i, chain-major), with the kernel a MALA
 * update runs.  EXTMCMC_EINVAL without a state or an installed user prior, EXTMCMC_EUNSUPPORTED for a
 * prior without gradient. */
int32_t extmcmc_eval_user_prior(extmcmc_t h, int32_t u, double *lp_out, double *grad_out);

/* Replaces RandomWalkUpdate(rw, coords; prior, adpt) src/updates.jl:170-182. */
int32_t extmcmc_set_update(extmcmc_t h, int32_t u, const extmcmc_update_t *upd);
/* theta[p * n_chains] chain-major SoA; replaces theta_init (src/run.jl:34-45).
 * Resets ll to -Inf (src/workspaces.jl:425), counters, moments and history.  The Philox
 * counters restart too: a caller that runs the sampler again on the same handle (warm-up,
 * then sampling) and wants fresh draws -- the reference advances a global RNG between runs --
 * calls extmcmc_set_seed first (the Python and Julia mirrors derive a new seed per run). */
int32_t extmcmc_set_state(extmcmc_t h, const double *theta);
/* Replaces the Philox key of the handle (cfg.seed). */
int32_t extmcmc_set_seed(extmcmc_t h, uint64_t seed);
/* HaarioTypeAdaptation's weight schedule lambda <- f(lambda, N, mcmc_iter) (the `f` keyword of
 * the constructor, adaptation.jl:385; applied by readjust!, :422-426).  lambda is shared by all
 * chains and N, mcmc_iter are schedule facts, so the library evaluates f on the HOST, on the
 * calling thread, inside extmcmc_run_block, once per readjustment of update u, and ships the
 * value with the step -- any closure works (Julia: @cfunction).  NULL restores the default
 * f = (lambda, N, iter) -> lambda. */
typedef double (*extmcmc_lambda_fn)(double lambda, int64_t N, int64_t mcmc_iter, void *user);
int32_t extmcmc_set_lambda_fn(extmcmc_t h, int32_t u, extmcmc_lambda_fn f, void *user);

/* ---- checkpoint / resume ---------------------------------------------------
 * Everything a later extmcmc_run_block depends on: chain state and log-likelihood, step sizes
 * (eps / Sigma_B and its factor / tau), adaptation counters, acceptance totals and rings, running
 * moments, Haario state, the lambda of every mixture walk, and the host bookkeeping (executed-step
 * count, rolling-acceptance tags).  The RNG has no state: a resumed run continues the same Philox
 * streams, so `run 2M` and `run M, save, load into a fresh handle with the same configuration,
 * updates and observations, run M with MCMCSchedule(...; start = ...)` (src/schedule.jl:28) are
 * bit-identical.  The history ring is not part of the blob.  _load checks the shape header (and, for
 * EXTMCMC_LAW_USER, a hash of the compiled law: a blob of another law is refused).
 * (Gradients and the data-sum cache of HIER_NORMAL are not part of the blob either: they are
 * recomputed on demand by the kernels that produced them, to the same bits.) */
int32_t extmcmc_checkpoint_size(extmcmc_t h, int64_t *bytes_out);
int32_t extmcmc_checkpoint_save(extmcmc_t h, void *blob, int64_t bytes);
int32_t extmcmc_checkpoint_load(extmcmc_t h, const void *blob, int64_t bytes);

/* ---- multi-rank (one process per GPU) ------------------------------------ */
/* Fills 128 bytes with an NCCL unique id (rank 0 calls it and ships the bytes
 * to the other ranks with any host transport, e.g. torch.distributed/gloo). */
int32_t extmcmc_comm_unique_id(uint8_t id_out[128]);
/* Joins the communicator; required before run_block under EXTMCMC_SHARD_OBS. */
int32_t extmcmc_comm_init(extmcmc_t h, const uint8_t id[128]);

/* Optional, on top of extmcmc_comm_init: the library's own exchange of the per-chain sums
 * (self-validating tagged cells stored straight into every peer's buffer over NVLink, polled and
 * combined in rank order inside the accept kernel: no fence, no flag) instead of ncclAllReduce on
 * the hot path.  Every rank exports a 64-byte CUDA IPC handle, the host ships
 * all of them to every rank (handles[world][64], rank order), every rank imports.  All ranks
 * must then call set_state / run_block in lock-step (they do: state and schedule are replicated). */
int32_t extmcmc_p2p_export(extmcmc_t h, uint8_t handle_out[64]);
int32_t extmcmc_p2p_import(extmcmc_t h, const uint8_t *handles);

/* ---- the hot path --------------------------------------------------------- */
/* Replaces the body of __run! (src/run.jl:70-82) for a run of consecutive
 * schedule elements: update_workspaces! (:101-112), update! (:197-208) =
 * proposal! + set_proposal! + compute_ll! + accept_reject! + update_stats!,
 * and update_adaptation! (:136-173).  Asynchronous on the handle's stream. */
int32_t extmcmc_run_block(extmcmc_t h, const extmcmc_step_t *steps, int32_t n_steps);
/* Same, with the randomness replayed: proposals[n_steps][p_u_max][n_chains]
 * (local proposal theta°_loc of the step's update, rows beyond its p_u unused)
 * and exp_draws[n_steps][n_chains] (the Exponential(1) draw of src/run.jl:278). */
int32_t extmcmc_run_block_replay(extmcmc_t h, const extmcmc_step_t *steps,
                                 int32_t n_steps, int32_t p_u_max,
                                 const double *proposals, const double *exp_draws);
/* Blocks until all queued work finished; returns EXTMCMC_EDOMAIN if any chain
 * left the law's domain since the last sync. */
int32_t extmcmc_sync(extmcmc_t h);

/* ---- read-back (host buffers caller-owned; NULL = skip) ------------------ */
int32_t extmcmc_get_state(extmcmc_t h, double *theta /* [p][C] */,
                          double *ll /* [C] */);
/* Rows of the executed-step sequence [seq_lo, seq_hi) counted from the last
 * set_state; mirrors state_history / state_proposal_history (src/workspaces.jl:
 * 157-189), ll_history (:413-434) and acceptance_history (:453-458).
 * theta, theta_prop: [n][p][C]; ll, ll_prop: [n][C]; accepted: [n][C] bytes. */
int32_t extmcmc_get_history(extmcmc_t h, int64_t seq_lo, int64_t seq_hi,
                            double *theta, double *theta_prop, double *ll,
                            double *ll_prop, uint8_t *accepted);
/* Asynchronous pair for overlapping the copy-back of block k with the execution of
 * block k+1 (callbacks fire only at save/print intervals, src/callbacks.jl:198-202,
 * 300-304, so histories need to reach the host only there).  _begin enqueues the
 * device->pinned-staging copy of rows [seq_lo, seq_hi) on a copy stream, ordered
 * after everything queued so far; _end waits for it and scatters the staging area
 * into the caller's buffers (same layouts as extmcmc_get_history).  One fetch may
 * be outstanding at a time. */
int32_t extmcmc_history_fetch_begin(extmcmc_t h, int64_t seq_lo, int64_t seq_hi);
int32_t extmcmc_history_fetch_end(extmcmc_t h, double *theta, double *theta_prop,
                                  double *ll, double *ll_prop, uint8_t *accepted);
/* GenericChainStats (src/chain_statistics.jl:16-66), per chain:
 * mean[p][C], cov[p][p][C] (column-major p x p, chain fastest),
 * rolling_ar[NU][C] (latest value per update), n_accept/n_prop[NU][C] totals. */
int32_t extmcmc_get_stats(extmcmc_t h, double *mean, double *cov,
                          double *rolling_ar, int64_t *n_accept, int64_t *n_prop);
/* Current step-size state of update u per chain: eps[p_u][C] (RW_UNIFORM),
 * Sigma_B[p_u*p_u][C] column-major (RW_GAUSS_MIX: gsn_B.Sigma after readjust!,
 * adaptation.jl:422-426), tau[1][C] (MALA). */
int32_t extmcmc_get_eps(extmcmc_t h, int32_t u, double *eps);
/* HaarioTypeAdaptation.mean [p_u][C] and .cov [p_u*p_u][C] (adaptation.jl:372-379). */
int32_t extmcmc_get_adapt_state(extmcmc_t h, int32_t u, double *mean, double *cov);
/* Evaluate the full-data log-likelihood of the current state of every chain
 * (one sweep, nothing else); ll_out[C].  Used by parity tests. */
int32_t extmcmc_eval_loglik(extmcmc_t h, double *ll_out);
/* Same plus the gradient d ll / d theta of all p parameters, grad_out[p][C] (laws with a
 * device gradient only).  The reference has only the hook for this:
 * compute_gradients_and_momenta! src/updates.jl:129-133, `grad ll` src/workspaces.jl:417. */
int32_t extmcmc_eval_grad(extmcmc_t h, double *ll_out, double *grad_out);

/* ---- measurement ---------------------------------------------------------- */
/* CUDA-event stopwatch on the handle's stream. */
int32_t extmcmc_timer_start(extmcmc_t h);
int32_t extmcmc_timer_stop(extmcmc_t h, float *ms_out);
/* Event pool on the handle's stream (idx in [0, 8192)): record now / elapsed ms between
 * two recorded events (synchronises on the later one).  Lets a caller time many
 * asynchronous blocks without a host sync in between. */
int32_t extmcmc_event_record(extmcmc_t h, int32_t idx);
int32_t extmcmc_event_elapsed(extmcmc_t h, int32_t idx_start, int32_t idx_stop, float *ms_out);
/* With cfg.instrument: accumulated device time and launch count of the
 * likelihood sweep kernel since the last call (resets the accumulators). */
int32_t extmcmc_get_sweep_time(extmcmc_t h, float *ms_total, int64_t *n_launches);
/* Kernels launched by this handle since creation. */
int64_t extmcmc_launch_count(extmcmc_t h);
/* Writes >= 256 MiB on the handle's stream to evict L2 (bench hygiene). */
int32_t extmcmc_flush_l2(extmcmc_t h);
/* FP64 FMA micro-benchmark on the handle's device: TFLOP/s (2 flop per FMA). */
int32_t extmcmc_measure_fp64_peak(extmcmc_t h, double *tflops_out);
/* FP64 tensor-core (DMMA m8n8k4) micro-benchmark: TFLOP/s. */
int32_t extmcmc_measure_dmma_peak(extmcmc_t h, double *tflops_out);
/* Name of the sweep kernel variant selected for the current shapes (user laws: user_chains_R1/R2/R4,
 * user_lanes). */
const char *extmcmc_sweep_variant_name(extmcmc_t h);

#ifdef __cplusplus
}
#endif
#endif /* EXTMCMC_H_ */
