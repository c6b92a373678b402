// Per-chain device functions of the transition step, shared by the per-step kernels
// (step_kernels.cu) and the persistent block kernels (block_kernels.cu).
//
// One thread owns a chain's scalar work; everything per-chain is SoA in global memory
// (q[k * C + c]), so the functions below STREAM over coordinates -- they take accessors instead of
// thread-local arrays, which keeps them free of local memory whatever p_u is.  The arithmetic
// (operand order, association) is the oracle's and therefore the reference's: translation units
// that include this header are compiled with -fmad=false, and the replay parity tests compare
// eps, running moments and trajectories bit-for-bit.
#pragma once
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>
#include "dev_state.cuh"
#include "philox.cuh"
#include "exchange.cuh"
#include "rw_draw.cuh"

namespace extmcmc {

constexpr double kLog2Pi = 1.8378770664093454835606594728112;
constexpr double kLogPi = 1.1447298858494001741434273513531;

// ---- accessors (StrideGet, CoordGet, MatRef: rw_draw.cuh) ------------------------------------
template <class G>
struct OffsetGet {
    G g;
    int off;
    __device__ __forceinline__ double operator()(int i) const { return g(off + i); }
};

// ---- compile-time specialisation ---------------------------------------------------------------
// The per-chain functions serve every transition kernel, prior family and law of the ABI.  Inlined
// into one step kernel that is ~40 000 SASS instructions, of which a chain's thread walks a few
// thousand, once per launch: the instruction fetch sits on the critical path (ncu, warm caches:
// 36-42 % of the worker warps' stall samples in the accept kernels are `no_inst`).  A StepSpec folds
// the dispatch at compile time.  SpecAny: everything dynamic (the general path).  SpecLean<LAW>: the
// law is LAW, every random-walk update of the handle is a UniformRandomWalk, every prior is one of
// Improper / ImproperPos / Normal and no update carries a HaarioTypeAdaptation -- the host checks
// this per handle (DevState.lean) and picks the instantiation; the arithmetic is the same code.
// The laws whose sweep finishes ll and gradient (law_self_finished) share SpecLean<LOGISTIC>: their
// step kernels do not depend on the law otherwise.
struct SpecAny {
    static constexpr int kLaw = -1;
    static constexpr bool kLean = false;
};
template <int LAW>
struct SpecLean {
    static constexpr int kLaw = LAW;
    static constexpr bool kLean = true;
};
template <class SP> __device__ __forceinline__ int sp_law(const DevState &d) { return SP::kLaw >= 0 ? SP::kLaw : d.law; }
template <class SP> __device__ __forceinline__ int sp_rw_kernel(const DevUpdate &u) {
    return SP::kLean ? (int)EXTMCMC_KERNEL_RW_UNIFORM : u.kernel;
}

// ---- priors: logpdf(prior, theta_loc) on the update's own coordinates (src/updates.jl:104,
//      src/priors.jl:18-39) ---------------------------------------------------------------------
template <bool LEAN = false, class Get>
__device__ __forceinline__ double log_prior_family(int kind, const double *pp, Get get, int n) {
    switch (kind) {
    case EXTMCMC_PRIOR_IMPROPER: return 0.0;  // priors.jl:19
    case EXTMCMC_PRIOR_IMPROPER_POS: {        // -sum(log.(th)), priors.jl:26
        double s = 0.0;
        for (int i = 0; i < n; ++i) s += log(get(i));
        return -s;
    }
    case EXTMCMC_PRIOR_NORMAL: {
        const double m = pp[0], sd = pp[1];
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double z = (get(i) - m) / sd;
            s += -(z * z + kLog2Pi) / 2.0 - log(sd);
        }
        return s;
    }
    case EXTMCMC_PRIOR_GAMMA: {
        if (LEAN) break;   // not a lean family: unreachable, the host never picks a lean kernel then
        const double k = pp[0], sc = pp[1];
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double x = get(i);
            if (!(x > 0.0)) return -INFINITY;
            s += -lgamma(k) - k * log(sc) + (k - 1.0) * log(x) - x / sc;
        }
        return s;
    }
    case EXTMCMC_PRIOR_UNIFORM: {
        if (LEAN) break;   // not a lean family: unreachable, the host never picks a lean kernel then
        const double a = pp[0], b = pp[1];
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double x = get(i);
            if (!(x >= a && x <= b)) return -INFINITY;
            s += -log(b - a);
        }
        return s;
    }
    case EXTMCMC_PRIOR_EXPONENTIAL: { /* Exponential(scale): log(rate) - rate x, rate = 1/scale; -Inf for x < 0 */
        if (LEAN) break;   // not a lean family: unreachable, the host never picks a lean kernel then
        const double rate = 1.0 / pp[0];
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double x = get(i);
            if (!(x >= 0.0)) return -INFINITY;
            s += log(rate) - rate * x;
        }
        return s;
    }
    case EXTMCMC_PRIOR_INV_GAMMA: { /* InverseGamma(a, sc): a log sc - lgamma(a) - (a + 1) log x - sc/x */
        if (LEAN) break;   // not a lean family: unreachable, the host never picks a lean kernel then
        const double a = pp[0], sc = pp[1];
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double x = get(i);
            if (!(x > 0.0)) return -INFINITY;
            s += a * log(sc) - lgamma(a) - (a + 1.0) * log(x) - sc / x;
        }
        return s;
    }
    case EXTMCMC_PRIOR_BETA: { /* Beta(a, b): (a-1) log x + (b-1) log1p(-x) - logbeta(a, b) on (0, 1) */
        if (LEAN) break;   // not a lean family: unreachable, the host never picks a lean kernel then
        const double a = pp[0], b = pp[1];
        const double lbeta = lgamma(a) + lgamma(b) - lgamma(a + b);
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double x = get(i);
            if (!(x > 0.0 && x < 1.0)) return -INFINITY;
            s += (a - 1.0) * log(x) + (b - 1.0) * log1p(-x) - lbeta;
        }
        return s;
    }
    case EXTMCMC_PRIOR_LOGNORMAL: { /* LogNormal(m, sd): logpdf(Normal(m, sd), log x) - log x */
        if (LEAN) break;   // not a lean family: unreachable, the host never picks a lean kernel then
        const double m = pp[0], sd = pp[1];
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double x = get(i);
            if (!(x > 0.0)) return -INFINITY;
            const double lx = log(x), z = (lx - m) / sd;
            s += (-(z * z + kLog2Pi) / 2.0 - log(sd)) - lx;
        }
        return s;
    }
    case EXTMCMC_PRIOR_CAUCHY: { /* Cauchy(m, sc): -(log1p(z^2) + log(pi) + log(sc)) */
        if (LEAN) break;   // not a lean family: unreachable, the host never picks a lean kernel then
        const double m = pp[0], sc = pp[1];
        double s = 0.0;
        for (int i = 0; i < n; ++i) {
            const double z = (get(i) - m) / sc;
            s += -(log1p(z * z) + kLogPi + log(sc));
        }
        return s;
    }
    }
    return NAN;
}

// logpdf(MvNormal(mu, L L'), x) by whitening z = inv(L) (x - mu); zs: this chain's scratch column
// (stride zstride).  L.get(r + k n): column-major lower factor.
template <class MuGet, class XGet>
__device__ __forceinline__ double mvn_logpdf_chol(const MatRef &L, int n, MuGet mu, XGet x, double *zs,
                                                  int64_t zstride) {
    double sq = 0.0, logdet = 0.0;
    for (int r = 0; r < n; ++r) {
        double a = x(r) - mu(r);
        for (int k = 0; k < r; ++k) a -= L.get(r + k * n) * zs[(int64_t)k * zstride];
        const double lrr = L.get(r + r * n);
        const double zr = a / lrr;
        zs[(int64_t)r * zstride] = zr;
        sq += zr * zr;
        logdet += log(lrr);
    }
    return -((double)n * kLog2Pi + 2.0 * logdet) / 2.0 - sq / 2.0;
}

template <class SP = SpecAny, class Get>
__device__ __forceinline__ double log_prior(const DevState &d, const DevUpdate &u, Get get, int64_t c) {
    if (SP::kLean) return log_prior_family<true>(u.prior, u.prior_params, get, u.n_coords);
    if (u.prior == EXTMCMC_PRIOR_MVNORMAL) {
        // StandardPrior(MvNormal(mu, Sigma)) on the whole coordinate block (priors.jl:35-39)
        const int n = u.n_coords;
        const MatRef L{const_cast<double *>(u.prior_dev) + n, 1};
        return mvn_logpdf_chol(L, n, StrideGet{u.prior_dev, 1}, get, d.gw + c, d.C);
    }
    if (u.prior != EXTMCMC_PRIOR_PRODUCT) return log_prior_family(u.prior, u.prior_params, get, u.n_coords);
    // ProductPrior (priors.jl:82-88): lp = 0.0; lp += logpdf(dist_k, th[idx_k])
    const int K = (int)u.prior_params[0];
    double lp = 0.0;
    int off = 0;
    for (int k = 0; k < K; ++k) {
        const double *f = u.prior_params + 1 + 4 * k;
        const int dim = (int)f[1];
        lp += log_prior_family((int)f[0], f + 2, OffsetGet<Get>{get, off}, dim);
        off += dim;
    }
    return lp;
}

// logpdf(rw::UniformRandomWalk, from, to) (random_walk.jl:88-94): only positive-
// constrained coordinates contribute, -log(2 eps_i) - log(to_i).
template <class EpsGet, class ToGet>
__device__ __forceinline__ double log_q_unif(const DevUpdate &u, EpsGet eps, ToGet to) {
    double s = 0.0;
    for (int i = 0; i < u.n_coords; ++i) {
        const double t = u.pos[i] ? (-log(2.0 * eps(i)) - log(to(i))) : 0.0;
        s = (i == 0) ? t : s + t;
    }
    return s;
}

// ---- Gaussian random walks (random_walk.jl:123-232) -------------------------------------------

// Lower Cholesky factor of Symmetric(S) (upper triangle of the column-major n x n S) written to L;
// false (and L[0] = NaN) when S is not positive definite.
__device__ __forceinline__ bool chol_lower_sym_upper(const MatRef &S, int n, const MatRef &L) {
    for (int j = 0; j < n; ++j) {
        double s = S.get(j + j * n);
        for (int k = 0; k < j; ++k) { const double l = L.get(j + k * n); s -= l * l; }
        if (!(s > 0.0) || isinf(s)) { L.set(0, NAN); return false; }
        const double ljj = sqrt(s);
        L.set(j + j * n, ljj);
        for (int i = j + 1; i < n; ++i) {
            double a = S.get(j + i * n);
            for (int k = 0; k < j; ++k) a -= L.get(i + k * n) * L.get(j + k * n);
            L.set(i + j * n, a / ljj);
        }
    }
    return true;
}

template <class G>
struct LogPosGet {            // remove_constraints on a copy: log of the positive coordinates
    G g;
    const uint8_t *pos;
    __device__ __forceinline__ double operator()(int i) const { const double x = g(i); return pos[i] ? log(x) : x; }
};

// logpdf(rw::GaussianRandomWalk, from, to) random_walk.jl:163-171, on transformed copies
template <class FromGet, class ToGet>
__device__ __forceinline__ double log_q_gauss(const DevState &d, const DevUpdate &u, const MatRef &L, FromGet from,
                                              ToGet to, int64_t c) {
    const int n = u.n_coords;
    double s = 0.0;
    for (int i = 0; i < n; ++i) if (u.pos[i]) s += log(to(i));
    const double logJ = -s;
    return mvn_logpdf_chol(L, n, LogPosGet<FromGet>{from, u.pos}, LogPosGet<ToGet>{to, u.pos}, d.gw + c, d.C) + logJ;
}

// q(from -> to) of a Gaussian walk (GaussianRandomWalkMix random_walk.jl:229-232: no log-sum-exp
// guard, as in the reference); NaN when a factor is missing (Sigma not positive definite)
template <class FromGet, class ToGet>
__device__ __forceinline__ double log_q_gauss_any(const DevState &d, const DevUpdate &u, double lambda, FromGet from,
                                                  ToGet to, int64_t c) {
    const double lpA = log_q_gauss(d, u, mat_LA(u), from, to, c);
    if (u.kernel == EXTMCMC_KERNEL_RW_GAUSS) return lpA;
    const double lpB = log_q_gauss(d, u, mat_LB(u, d.C, c), from, to, c);
    return log((1.0 - lambda) * exp(lpA) + lambda * exp(lpB));
}

// ---- per-chain law constants of a parameter vector ---------------------------------------------
//   GSN_IID_1D: lawc = { mu, c0 = -(log 2pi + 2 log sqrt(var))/2, 1/(2 var) },
//               ll = N c0 - S/(2 var),  S = sum (x - mu)^2     (gsn_target.jl:15-29, d = 1)
//   GSN_MV(d):  lawc = { mu[d], W = inv(L) lower-tri row-major, c0 },  Sigma = L L' built from the
//               UPPER triangle of the d x d block of theta (Symmetric(triu(S)), gsn_target.jl:19);
//               ll = N c0 - S/2,  S = sum |W (x - mu)|^2,  c0 = -(d log 2pi + 2 sum log L_ii)/2
template <class SP = SpecAny>
__device__ __forceinline__ void law_prepare(const DevState &d, int64_t c, const double *full,
                                            int64_t stride) {
    const int law = sp_law<SP>(d);
    if (law == EXTMCMC_LAW_GSN_IID_1D) {
        const double mu = full[0], var = full[stride];
        double c0, inv2;
        if (!(var > 0.0) || isinf(var)) {
            c0 = NAN; inv2 = NAN;
            *d.err_flag = 1;
        } else {
            c0 = -(kLog2Pi + 2.0 * log(sqrt(var))) / 2.0;
            inv2 = 0.5 / var;
        }
        d.lawc[c] = mu;
        d.lawc[d.C + c] = c0;
        d.lawc[2 * d.C + c] = inv2;
    } else if (law == EXTMCMC_LAW_HIER_NORMAL) {
        // no constants: the sweep reads theta_1..G straight from the state array it is given
        const double tau = full[(int64_t)(d.G + 1) * stride];
        if (!(tau > 0.0) || isinf(tau)) *d.err_flag = 1;
    } else if (law == EXTMCMC_LAW_GSN_MV) {
        const int n = d.obs_dim;
        const int64_t C = d.C;
        double *L = d.mv_L + c;                       // L[i][k] at (i n + k) C
        double *W = d.lawc + (int64_t)n * C + c;      // W[i][j] (j <= i) at (i (i + 1) / 2 + j) C
        bool bad = false;
        // A[i][j] (i >= j) = theta[n + j + i*n]: entry (row j, col i) of the column-major block
        for (int j = 0; j < n && !bad; ++j) {
            double s = full[(int64_t)(n + j + j * n) * stride];
            for (int k = 0; k < j; ++k) { const double l = L[(int64_t)(j * n + k) * C]; s -= l * l; }
            if (!(s > 0.0) || isinf(s)) { bad = true; break; }
            const double ljj = sqrt(s);
            L[(int64_t)(j * n + j) * C] = ljj;
            for (int i = j + 1; i < n; ++i) {
                double a = full[(int64_t)(n + j + i * n) * stride];
                for (int k = 0; k < j; ++k) a -= L[(int64_t)(i * n + k) * C] * L[(int64_t)(j * n + k) * C];
                L[(int64_t)(i * n + j) * C] = a / ljj;
            }
        }
        double logdet = 0.0;
        if (!bad) {
            // W = inv(L): forward substitution column by column
            for (int j = 0; j < n; ++j) {
                const double ljj = L[(int64_t)(j * n + j) * C];
                W[(int64_t)(j * (j + 1) / 2 + j) * C] = 1.0 / ljj;
                for (int i = j + 1; i < n; ++i) {
                    double a = 0.0;
                    for (int k = j; k < i; ++k) a -= L[(int64_t)(i * n + k) * C] * W[(int64_t)(k * (k + 1) / 2 + j) * C];
                    W[(int64_t)(i * (i + 1) / 2 + j) * C] = a / L[(int64_t)(i * n + i) * C];
                }
                logdet += log(ljj);
            }
        } else {
            *d.err_flag = 1;
            for (int w = 0; w < n * (n + 1) / 2; ++w) W[(int64_t)w * C] = NAN;
        }
        for (int j = 0; j < n; ++j) d.lawc[(int64_t)j * C + c] = full[(int64_t)j * stride];
        d.lawc[(int64_t)(d.lawc_k - 1) * C + c] = bad ? NAN : -((double)n * kLog2Pi + 2.0 * logdet) / 2.0;
    }
}

// th: this chain's parameter vector the sums were computed for (stride C)
template <class SP = SpecAny>
__device__ __forceinline__ double law_finalize(const DevState &d, int64_t c, double S, const double *th) {
    const int law = sp_law<SP>(d);
    if (law_self_finished(law)) return S;  // the sweep finished ll itself
    if (law == EXTMCMC_LAW_GSN_IID_1D)  // N*c0 - S/(2 var)
        return (double)d.n_obs_total * d.lawc[d.C + c] - S * d.lawc[2 * d.C + c];
    if (law == EXTMCMC_LAW_HIER_NORMAL) {
        // sum_gj logN(y_gj; th_g, 1) + sum_g logN(th_g; mu, tau^2)
        const int G = d.G;
        const double mu = th[(int64_t)G * d.C], tau = th[(int64_t)(G + 1) * d.C];
        if (!(tau > 0.0) || isinf(tau)) return NAN;
        double dev2 = 0.0;
        for (int g = 0; g < G; ++g) { const double dv = th[(int64_t)g * d.C] - mu; dev2 += dv * dv; }
        return -0.5 * (double)d.n_obs_total * kLog2Pi - S / 2.0 +
               (double)G * (-0.5 * kLog2Pi - log(tau)) - dev2 / (2.0 * tau * tau);
    }
    return (double)d.n_obs_total * d.lawc[(int64_t)(d.lawc_k - 1) * d.C + c] - S / 2.0;
}

// The schedule element and its update entry are read by every thread dozens of times;
// stage them in shared memory once per CTA (a dependent chain of global loads otherwise).
struct StepCtx {
    StepDesc sd;
    DevUpdate u;
};
// tid / nthreads: index and size of the thread group that shares `ctx`; the caller synchronises the
// group between the two phases (sync()) and after the call
template <class Sync>
__device__ __forceinline__ void load_step_ctx(StepCtx *ctx, const DevState &d, const StepDesc *descs, int k,
                                              int tid, int nthreads, Sync sync) {
    static_assert(sizeof(StepDesc) % 4 == 0 && sizeof(DevUpdate) % 4 == 0, "word copies");
    const uint32_t *src = reinterpret_cast<const uint32_t *>(descs + k);
    uint32_t *dst = reinterpret_cast<uint32_t *>(&ctx->sd);
    for (int i = tid; i < (int)(sizeof(StepDesc) / 4); i += nthreads) dst[i] = src[i];
    sync();
    const uint32_t *us = reinterpret_cast<const uint32_t *>(d.upd + ctx->sd.pidx);
    uint32_t *ud = reinterpret_cast<uint32_t *>(&ctx->u);
    for (int i = tid; i < (int)(sizeof(DevUpdate) / 4); i += nthreads) ud[i] = us[i];
    sync();
}
struct CtaSync { __device__ __forceinline__ void operator()() const { __syncthreads(); } };

// ---------------------------------------------------------------------------------
// proposal!  (src/updates.jl:191-196, rand(::UniformRandomWalk) random_walk.jl:65-73)
//     + set_proposal! (src/run.jl:221-240): writes the local and the full proposal and the law
//     constants the sweep consumes.
// ---------------------------------------------------------------------------------
// Two halves, so that a step kernel can run them on a warp of their own next to the bookkeeping of
// the step just decided: propose_draw reads the committed state and writes prop_loc / n_used;
// propose_set writes prop_full and the law constants (the bookkeeping must have read prop_full for
// its history row by then).  propose_chain = both, back to back.
template <class SP = SpecAny>
__device__ __forceinline__ void propose_draw(const DevState &d, const StepDesc &sd, const DevUpdate &u, int64_t c) {
    rw_draw(d, sd, u, c, sp_rw_kernel<SP>(u), [&](const StrideGet &prop) { return log_prior<SP>(d, u, prop, c); });
}

template <class SP = SpecAny>
__device__ __forceinline__ void propose_set(const DevState &d, const DevUpdate &u, int64_t c) {
    const int n = u.n_coords;
    const int64_t C = d.C;
    const double *pl = d.prop_loc + c;
    // full proposal = current state with the update's coordinates replaced (run.jl:237-239);
    // loads in batches of 4 ahead of the stores (the arrays may alias as far as the compiler knows)
    for (int j0 = 0; j0 < d.p; j0 += 4) {
        double t[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) if (j0 + q < d.p) t[q] = d.theta[(int64_t)(j0 + q) * C + c];
#pragma unroll
        for (int q = 0; q < 4; ++q) if (j0 + q < d.p) d.prop_full[(int64_t)(j0 + q) * C + c] = t[q];
    }
    for (int i = 0; i < n; ++i) d.prop_full[(int64_t)u.coords[i] * C + c] = pl[(int64_t)i * C];
    law_prepare<SP>(d, c, d.prop_full + c, C);
}

template <class SP = SpecAny>
__device__ __forceinline__ void propose_chain(const DevState &d, const StepDesc &sd, const DevUpdate &u, int64_t c) {
    propose_draw<SP>(d, sd, u, c);
    propose_set<SP>(d, u, c);
}

// Cooperative covariance update for models with more than a handful of parameters (cfg 4: p = 10,
// full p x p covariance).  A thread group owns nch chains; the chain's own thread stages the
// committed state, the OLD running mean and the NEW running mean in shared memory, then, after a
// group barrier, ALL threads of the group update the nch x p x p covariance entries -- same
// arithmetic, one entry per thread per pass, coalesced along the chain axis -- instead of one
// thread walking p^2 dependent loads.
constexpr int kCoopP = 32;   // largest p served this way
struct CoopStage {
    double *t;   // [p][nch] committed state
    double *m;   // [p][nch] running mean before this step; nullptr unless the full covariance is kept
    double *mn;  // [p][nch] running mean after this step (spares two divisions per covariance entry)
    int nch, ch;
};

__device__ __forceinline__ void update_cov_coop(const DevState &d, int64_t N, int64_t c0, int nch, const double *sh_t,
                                                const double *sh_m, const double *sh_n, int tid, int nt) {
    const int p = d.p;
    const int64_t C = d.C;
    const double f_old = (double)(N - 1) / (double)N;
    const double f_new = (double)(N + 1) / (double)N;
    // nt is a multiple of nch: a thread keeps its chain and walks the entries e = a + b p with stride
    // nt / nch; (a, b) advance incrementally (no integer division by the run-time p in the loop)
    if (nt % nch != 0) {   // general thread-group shape (block kernels): flat index, divisions
        const int total = nch * p * p;
        for (int i = tid; i < total; i += nt) {
            const int ch = i % nch, e = i / nch;
            if (c0 + ch >= C) continue;
            const int a = e % p, b = e / p;
            const double ta = sh_t[a * nch + ch], tb = sh_t[b * nch + ch];
            const double ma_old = sh_m[a * nch + ch], mb_old = sh_m[b * nch + ch];
            const double ma_new = sh_n[a * nch + ch], mb_new = sh_n[b * nch + ch];
            const double old_sum_sq = f_old * d.cov[(int64_t)e * C + c0 + ch] + ma_old * mb_old;
            const double new_sum_sq = old_sum_sq + (ta * tb) / (double)N;
            d.cov[(int64_t)e * C + c0 + ch] = new_sum_sq - f_new * (ma_new * mb_new);
        }
        return;
    }
    // The recursion is symmetric in (a, b) -- every product in it commutes, and the matrix starts
    // symmetric -- so entry (b, a) is bit for bit entry (a, b): only the p (p + 1) / 2 entries with
    // a <= b are computed (one division each) and stored to both places.  They are walked column by
    // column, e = a + b (b + 1) / 2.
    const int ch = tid % nch, es = nt / nch, tri = p * (p + 1) / 2;
    const bool live = c0 + ch < C;
    int e = tid / nch, a = e, b = 0;
    while (a > b) { a -= b + 1; ++b; }
    for (; e < tri; ) {
        double cv[4];
        int ea[4], eb[4], ee[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            ee[q] = e; ea[q] = a; eb[q] = b;
            cv[q] = (e < tri && live) ? d.cov[(int64_t)(a + b * p) * C + c0 + ch] : 0.0;
            e += es; a += es;
            while (a > b) { a -= b + 1; ++b; }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (ee[q] < tri && live) {
                const double ta = sh_t[ea[q] * nch + ch], tb = sh_t[eb[q] * nch + ch];
                const double ma_old = sh_m[ea[q] * nch + ch], mb_old = sh_m[eb[q] * nch + ch];
                const double ma_new = sh_n[ea[q] * nch + ch], mb_new = sh_n[eb[q] * nch + ch];
                const double old_sum_sq = f_old * cv[q] + ma_old * mb_old;
                const double new_sum_sq = old_sum_sq + (ta * tb) / (double)N;
                const double v = new_sum_sq - f_new * (ma_new * mb_new);
                d.cov[(int64_t)(ea[q] + eb[q] * p) * C + c0 + ch] = v;
                if (ea[q] != eb[q]) d.cov[(int64_t)(eb[q] + ea[q] * p) * C + c0 + ch] = v;
            }
        }
    }
}

// ---------------------------------------------------------------------------------
// What follows an accept/reject decision, shared by the random-walk and MALA paths:
// register_accept_reject_results! (src/run.jl:299-335) + set_chain_param! (:312-320, the
// caller has already committed theta) + update_stats! (src/chain_statistics.jl:41-66) +
// update_adaptation! (src/run.jl:136-173, src/transition_kernels/adaptation.jl:273-329).
// n_eps = entries of the update's step-size vector (p_u for the uniform walk, 1 for MALA).
// ---------------------------------------------------------------------------------
// Two halves (a step kernel may run the next proposal on another warp in between, see propose_draw):
// post_decision_moments -- history row + running moments, reads theta / prop_full / mean / cov;
// post_decision_counters -- rolling acceptance rate, totals, adaptation.  post_decision = both.
// HIST / MOM select the two parts of the first half: the history row (+ the carried ll) and the running
// moments.  A step kernel that DEFERS its bookkeeping writes only the history row (the full proposal is
// about to be overwritten by the next one); moments and counters are then run by the next step kernel
// in its prologue, behind the next sweep (step_kernels.cu, "deferred bookkeeping").
// grp / n_grp: the per-parameter part (history row, staging, mean, diagonal statistics) is independent from
// parameter to parameter, so several threads may share a chain -- thread `grp` of `n_grp` takes the
// parameters [4 grp, 4 grp + 4), [4 (grp + n_grp), ...); the per-chain scalars belong to grp 0.  Only where
// nothing else follows the loop: not with the thread-alone full covariance (stats_mode 0 without cs->m).
template <class SP = SpecAny, bool HIST = true, bool MOM = true>
__device__ __forceinline__ void post_decision_moments(const DevState &d, const StepDesc &sd, int64_t c, bool accepted,
                                                      double ll_new, double ll_prop, const CoopStage *cs = nullptr,
                                                      int grp = 0, int n_grp = 1) {
    const int64_t C = d.C;
    if (HIST && grp == 0) d.ll[c] = ll_new;
    // history row (state_history / state_proposal_history / ll_history / acceptance_history)
    const int64_t slot = sd.seq % d.H;
    const int64_t hc = d.g0 + c;       // this chain's column in the arrays that stay global
    const int64_t N = sd.stat_n;
    const double f_old = (double)(N - 1) / (double)N;
    const double f_mean = (double)N / (double)(N + 1);
    const double f_new = (double)(N + 1) / (double)N;
    const bool coop_full = MOM && cs && cs->m;        // full covariance left to update_cov_coop
    const bool diag = MOM && d.stats_mode == 1;
    // History row, staging and -- diagonal statistics / cooperative path -- update_stats!
    // (chain_statistics.jl:46-51, verbatim arithmetic); loads in batches of 4 ahead of the stores
    // (the stores may alias the loads as far as the compiler knows, so a plain loop serialises).
    for (int j0 = 4 * grp; j0 < d.p; j0 += 4 * n_grp) {
        double t[4], pr[4], m[4], cv[4];
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (j0 + q < d.p) {
                t[q] = d.theta[(int64_t)(j0 + q) * C + c];
                if (HIST) pr[q] = d.prop_full[(int64_t)(j0 + q) * C + c];
                if (coop_full || diag) m[q] = d.mean[(int64_t)(j0 + q) * C + c];
                if (diag) cv[q] = d.cov[(int64_t)(j0 + q) * C + c];
            }
#pragma unroll
        for (int q = 0; q < 4; ++q)
            if (j0 + q < d.p) {
                const int j = j0 + q;
                if (HIST) {
                    d.h_theta[(slot * d.p + j) * d.gC + hc] = t[q];
                    d.h_prop[(slot * d.p + j) * d.gC + hc] = pr[q];
                }
                if (MOM && cs) cs->t[j * cs->nch + cs->ch] = t[q];
                if (coop_full || diag) {
                    const double m_new = m[q] * f_mean + t[q] / (double)(N + 1);
                    if (coop_full) { cs->m[j * cs->nch + cs->ch] = m[q]; cs->mn[j * cs->nch + cs->ch] = m_new; }
                    if (diag) {
                        const double old_sum_sq = f_old * cv[q] + m[q] * m[q];
                        const double new_sum_sq = old_sum_sq + (t[q] * t[q]) / (double)N;
                        d.cov[(int64_t)j * C + c] = new_sum_sq - f_new * (m_new * m_new);
                    }
                    d.mean[(int64_t)j * C + c] = m_new;
                }
            }
    }
    if (HIST && grp == 0) {
        d.h_ll[slot * d.gC + hc] = ll_new;
        d.h_llp[slot * d.gC + hc] = ll_prop;
        d.h_acc[slot * d.gC + hc] = accepted ? 1 : 0;
    }

    // full covariance by this thread alone (more than kCoopP parameters, or no spare threads)
    if (MOM && d.stats_mode == 0 && !coop_full && grp == 0) {
        const int p = d.p;
        // covariance first (it needs the old mean), column by column
        for (int b = 0; b < p; ++b) {
            const double tb = d.theta[(int64_t)b * C + c];
            const double mb_old = d.mean[(int64_t)b * C + c];
            const double mb_new = mb_old * f_mean + tb / (double)(N + 1);
            for (int a = 0; a < p; ++a) {
                const double ta = d.theta[(int64_t)a * C + c];
                const double ma_old = d.mean[(int64_t)a * C + c];
                const double ma_new = ma_old * f_mean + ta / (double)(N + 1);
                const int64_t idx = ((int64_t)(a + b * p)) * C + c;
                const double old_sum_sq = f_old * d.cov[idx] + ma_old * mb_old;
                const double new_sum_sq = old_sum_sq + (ta * tb) / (double)N;
                d.cov[idx] = new_sum_sq - f_new * (ma_new * mb_new);
            }
        }
        for (int a = 0; a < p; ++a) {
            const int64_t idx = (int64_t)a * C + c;
            d.mean[idx] = d.mean[idx] * f_mean + d.theta[idx] / (double)(N + 1);
        }
    }
}

template <class SP = SpecAny>
__device__ __forceinline__ void post_decision_counters(const DevState &d, const StepDesc &sd, const DevUpdate &u,
                                                       int64_t c, bool accepted, int n_eps) {
    const int64_t C = d.C;
    const int64_t N = sd.stat_n;
    // rolling acceptance rate (chain_statistics.jl:53-64)
    {
        const int W = d.W;
        const double ra_prev = sd.ra_prev_valid ? u.ra_val[c] : 0.0;
        const int64_t rslot = sd.mcmciter % W;
        const int acc_out = sd.acc_out_valid ? (int)u.acc_ring[rslot * C + c] : 0;
        const int64_t mn = (int64_t)W < N ? (int64_t)W : N;
        u.ra_val[c] = (ra_prev * (double)W + (double)((int)accepted - acc_out)) / (double)mn;
        u.acc_ring[rslot * C + c] = accepted ? 1 : 0;
    }

    // update_adaptation! -- only the update whose turn it is registers (run.jl:176-177)
    u.tot_prop[c] += 1;
    u.tot_acc[c] += accepted ? 1 : 0;
    if (u.adapt_kind == EXTMCMC_ADAPT_UNIF_RW || u.adapt_kind == EXTMCMC_ADAPT_MALA) {
        int32_t prop_n = u.adapt_prop[c] + 1;                      // register! :292-295
        int32_t acc_n = u.adapt_acc[c] + (accepted ? 1 : 0);
        if (prop_n >= u.adapt_every_k) {                           // time_to_update :302-304
            const double r = (double)sd.mcmciter / (double)u.adapt_every_k - u.offset;
            const double delta = u.scale / sqrt(r > 1.0 ? r : 1.0);  // compute_delta :312-319
            const double a_r = (double)acc_n / (double)prop_n;       // acceptance_rate :242-244
            prop_n = 0; acc_n = 0;                                   // reset! :263-266
            const double sgn = (a_r > u.target) ? 1.0 : -1.0;
            for (int i = 0; i < n_eps; ++i) {                        // compute_eps :326-329
                double e = u.eps[(int64_t)i * C + c] + sgn * delta;
                e = e < u.vmax ? e : u.vmax;
                e = e > u.vmin ? e : u.vmin;
                u.eps[(int64_t)i * C + c] = e;
            }
        }
        u.adapt_prop[c] = prop_n;
        u.adapt_acc[c] = acc_n;
    }
    // HaarioTypeAdaptation registers on EVERY update step of ANY update (adaptation.jl:399-414),
    // on that update's view of the (already committed) global state, log-transformed copy.
    if (!SP::kLean && d.n_haario > 0) {
        for (int v = 0; v < d.NU; ++v) {
            const DevUpdate &w = (v == sd.pidx) ? u : d.upd[v];
            if (w.adapt_kind != EXTMCMC_ADAPT_HAARIO) continue;
            const int m = w.n_coords;
            double *t = d.gw + (int64_t)d.gw_n * C + c;        // transformed sub-state
            double *om = d.gw + (int64_t)2 * d.gw_n * C + c;   // mean before this registration
            const int64_t hn = sd.stat_n;  // adpt.N: starts at 1, +1 per registration = per executed step
            const double hf_old = (double)(hn - 1) / (double)hn, hf_mean = (double)hn / (double)(hn + 1);
            const double hf_new = (double)(hn + 1) / (double)hn;
            for (int i = 0; i < m; ++i) {
                const double x = d.theta[(int64_t)w.coords[i] * C + c];
                const double ti = w.pos[i] ? log(x) : x;
                const double omi = w.hmean[(int64_t)i * C + c];
                t[(int64_t)i * C] = ti;
                om[(int64_t)i * C] = omi;
                w.hmean[(int64_t)i * C + c] = omi * hf_mean + ti / (double)(hn + 1);
            }
            const bool ready = (v == sd.pidx) && sd.haario_ready;
            for (int b = 0; b < m; ++b)
                for (int a = 0; a < m; ++a) {
                    const int64_t idx = (int64_t)(a + b * m) * C + c;
                    const double old_sum_sq = hf_old * w.hcov[idx] + om[(int64_t)a * C] * om[(int64_t)b * C];
                    const double new_sum_sq = old_sum_sq + (t[(int64_t)a * C] * t[(int64_t)b * C]) / (double)hn;
                    const double cv = new_sum_sq - hf_new * (w.hmean[(int64_t)a * C + c] * w.hmean[(int64_t)b * C + c]);
                    w.hcov[idx] = cv;
                    // readjust!(rw::GaussianRandomWalkMix, ...) adaptation.jl:422-426
                    if (ready) w.sigB[idx] = (2.38 * 2.38) / (double)m * cv;
                }
            // the factor of the new Sigma_B, cached for the proposals and densities to come
            if (ready) chol_lower_sym_upper(MatRef{w.sigB + c, C}, m, MatRef{w.LB + c, C});
        }
    }
}

template <class SP = SpecAny>
__device__ __forceinline__ void post_decision(const DevState &d, const StepDesc &sd, const DevUpdate &u,
                                              int64_t c, bool accepted, double ll_new, double ll_prop,
                                              int n_eps, const CoopStage *cs = nullptr) {
    post_decision_moments<SP>(d, sd, c, accepted, ll_new, ll_prop, cs);
    post_decision_counters<SP>(d, sd, u, c, accepted, n_eps);
}

__device__ __forceinline__ double draw_exp(const DevState &d, const StepDesc &sd, int64_t c) {
    if (d.rng_mode == EXTMCMC_RNG_REPLAY) return d.rp_exp[(int64_t)sd.replay_row * d.gC + d.g0 + c];
    ChainStepStream rng(d.seed, (uint64_t)(d.chain_offset + c), sd.mcmciter, sd.pidx, d.n_used[c]);
    return -log(rng.next());  // rand(Exponential(1.0)), run.jl:278
}

// ---------------------------------------------------------------------------------
// accept_reject! (src/run.jl:268-281) for the random-walk updates, in two halves: everything that
// does not depend on the proposal's log-likelihood (transition densities, priors, the Exp(1)
// draw), and the decision + commit once the sweep's sum S is known.
// ---------------------------------------------------------------------------------
struct RwPre {
    double ll_cur, q_back, q_fwd, lp_prop, lp_cur, E;
};

template <class SP = SpecAny>
__device__ __forceinline__ RwPre rw_accept_prologue(const DevState &d, const StepDesc &sd, const DevUpdate &u,
                                                    int64_t c) {
    const int kern = sp_rw_kernel<SP>(u);
    const int64_t C = d.C;
    const CoordGet th{d.theta + c, u.coords, C};
    const StrideGet prop{d.prop_loc + c, C};
    RwPre r;
    // update_workspaces! (run.jl:101-112): ll of the previously executed update; on the
    // very first element it is still the initial -Inf (workspaces.jl:425)
    r.ll_cur = sd.first ? -INFINITY : d.ll[c];
    if (kern == EXTMCMC_KERNEL_RW_UNIFORM) {
        const StrideGet eps{u.eps + c, C};
        r.q_back = log_q_unif(u, eps, th);    // theta° -> theta
        r.q_fwd = log_q_unif(u, eps, prop);   // theta -> theta°
    } else {
        const bool ok = !isnan(u.LA[0]) && (kern != EXTMCMC_KERNEL_RW_GAUSS_MIX || !isnan(u.LB[c]));
        if (!ok) {
            *d.err_flag = 1;
            r.q_back = NAN;
            r.q_fwd = 0.0;
        } else {
            r.q_back = log_q_gauss_any(d, u, sd.lambda, prop, th, c);   // theta° -> theta
            r.q_fwd = log_q_gauss_any(d, u, sd.lambda, th, prop, c);    // theta -> theta°
        }
    }
    if (!SP::kLean && u.prior == EXTMCMC_PRIOR_USER) {
        // a user-defined prior: its kernel drew the proposal and left both terms in prior_dev ([2][C])
        r.lp_prop = u.prior_dev[c];
        r.lp_cur = u.prior_dev[C + c];
    } else {
        r.lp_prop = log_prior<SP>(d, u, prop, c);
        r.lp_cur = log_prior<SP>(d, u, th, c);
    }
    r.E = draw_exp(d, sd, c);
    return r;
}

// S: the sweep's sum for the proposal.  Returns the decision; the chain state, history, running
// moments and adaptation state are updated.
struct Decision {
    bool accepted;
    double ll_new, ll_prop;
};
template <class SP = SpecAny>
__device__ __forceinline__ Decision rw_decide_commit(const DevState &d, const DevUpdate &u, int64_t c, const RwPre &r,
                                                     double S) {
    const int64_t C = d.C;
    const int n = u.n_coords;
    const double ll_prop = law_finalize<SP>(d, c, S, d.prop_full + c);
    // llr, strictly left to right (run.jl:271-277)
    double llr = ll_prop - r.ll_cur;
    llr = llr + r.q_back;
    llr = llr - r.q_fwd;
    llr = llr + r.lp_prop;
    llr = llr - r.lp_cur;
    const bool accepted = r.E > -llr;  // NaN compares false -> reject
    const double ll_new = accepted ? ll_prop : r.ll_cur;
    if (accepted)
        for (int i = 0; i < n; ++i) d.theta[(int64_t)u.coords[i] * C + c] = d.prop_loc[(int64_t)i * C + c];
    return Decision{accepted, ll_new, ll_prop};
}
template <class SP = SpecAny>
__device__ __forceinline__ int rw_n_eps(const DevUpdate &u) {
    return sp_rw_kernel<SP>(u) == EXTMCMC_KERNEL_RW_UNIFORM ? u.n_coords : 0;
}
template <class SP = SpecAny>
__device__ __forceinline__ bool rw_accept_finish(const DevState &d, const StepDesc &sd, const DevUpdate &u, int64_t c,
                                                 const RwPre &r, double S, const CoopStage *cs = nullptr) {
    const Decision dec = rw_decide_commit<SP>(d, u, c, r, S);
    post_decision<SP>(d, sd, u, c, dec.accepted, dec.ll_new, dec.ll_prop, rw_n_eps<SP>(u), cs);
    return dec.accepted;
}

// ---------------------------------------------------------------------------------
// Gradient path (MALAUpdate; the reference only has the hooks: MCMCGradientBasedUpdate
// src/types.jl:24, compute_gradients_and_momenta! src/updates.jl:129-133 called at
// src/run.jl:110,259, the `∇ll` buffer src/workspaces.jl:417).
//
// grad_finalize_chain: fixed-order reduction of the sweep's partial sums per chain (and
// per observation group), then ll and d ll / d theta for ALL p parameters.
//   GSN_IID_1D : d/dmu = T/var, d/dvar = -N/(2 var) + S/(2 var^2)
//   HIER_NORMAL: theta = [th_1..th_G, mu, tau], y_gj ~ N(th_g, 1), th_g ~ N(mu, tau^2) (the
//                hierarchical term lives in the law because priors only see their own
//                coordinates, src/run.jl:374-385):
//                d/dth_g = T_g - (th_g - mu)/tau^2, d/dmu = sum_g (th_g - mu)/tau^2,
//                d/dtau = -G/tau + sum_g (th_g - mu)^2 / tau^3
// ---------------------------------------------------------------------------------
template <class SP = SpecAny>
__device__ __forceinline__ void grad_finalize_chain(const DevState &d, int64_t c, const double *__restrict__ src,
                                                    double *__restrict__ ll_out, double *__restrict__ grad_out) {
    const int law = sp_law<SP>(d);
    const int64_t C = d.C, PC = d.gC;
    const double *part = d.partial + d.g0 + c;   // this chain's column of partial[2][G*S][gC]
    const int G = d.G, S = d.S;
    const int64_t rows = (int64_t)G * S;
    if (law == EXTMCMC_LAW_GSN_IID_1D) {
        double s2 = 0.0, s1 = 0.0;
        for (int i = 0; i < S; ++i) { s2 += __ldcg(part + (int64_t)i * PC); s1 += __ldcg(part + (rows + i) * PC); }
        const double var = src[C + c];
        ll_out[c] = law_finalize<SP>(d, c, s2, src + c);
        grad_out[c] = s1 / var;
        grad_out[C + c] = -(double)d.n_obs_total / (2.0 * var) + s2 / (2.0 * var * var);
    } else if (law == EXTMCMC_LAW_HIER_NORMAL) {
        const double mu = src[(int64_t)G * C + c], tau = src[(int64_t)(G + 1) * C + c];
        if (!(tau > 0.0) || isinf(tau)) *d.err_flag = 1;   // the current state never went through law_prepare
        const double it2 = 1.0 / (tau * tau);
        double s2_tot = 0.0, dmu = 0.0, dev2 = 0.0;
        for (int g = 0; g < G; ++g) {
            double s2 = 0.0, s1 = 0.0;
            for (int i = 0; i < S; ++i) {
                s2 += __ldcg(part + ((int64_t)g * S + i) * PC);
                s1 += __ldcg(part + (rows + (int64_t)g * S + i) * PC);
            }
            s2_tot += s2;
            const double dv = src[(int64_t)g * C + c] - mu;
            grad_out[(int64_t)g * C + c] = s1 - dv * it2;
            dmu += dv * it2;
            dev2 += dv * dv;
        }
        grad_out[(int64_t)G * C + c] = dmu;
        grad_out[(int64_t)(G + 1) * C + c] = -(double)G / tau + dev2 * it2 / tau;
        ll_out[c] = law_finalize<SP>(d, c, s2_tot, src + c);
    }
}

// d log prior / d theta_i for the priors that have one on the device
__device__ __forceinline__ double prior_grad(const DevUpdate &u, double th) {
    if (u.prior == EXTMCMC_PRIOR_NORMAL) return -(th - u.prior_params[0]) / (u.prior_params[1] * u.prior_params[1]);
    return 0.0;  // ImproperPrior
}
__device__ __forceinline__ double prior_logpdf1(const DevUpdate &u, double th) {
    if (u.prior == EXTMCMC_PRIOR_NORMAL) {
        const double z = (th - u.prior_params[0]) / u.prior_params[1];
        return -(z * z + kLog2Pi) / 2.0 - log(u.prior_params[1]);
    }
    return 0.0;
}

// d log prior / d theta_i of a MALA update: the built-in families, or -- a user-defined prior, general
// path only -- what its gradient kernel left in prior_dev: [2][1 + p_u][C], state s = 0 the current one,
// s = 1 the proposal, row 0 the log prior and row 1 + i its derivative in coordinate i
template <class SP>
__device__ __forceinline__ double mala_prior_grad(const DevUpdate &u, double th, int64_t C, int64_t c, int s, int i) {
    if (!SP::kLean && u.prior == EXTMCMC_PRIOR_USER) return u.prior_dev[((int64_t)s * (1 + u.n_coords) + 1 + i) * C + c];
    return prior_grad(u, th);
}

// MALA proposal  theta° = theta + (tau^2/2) g(theta) + tau z,  g = grad(ll + log prior)
template <class SP = SpecAny>
__device__ __forceinline__ void mala_propose_chain(const DevState &d, const StepDesc &sd, const DevUpdate &u, int64_t c) {
    const int64_t C = d.C;
    const int n = u.n_coords;
    const double tau = u.eps[c], h2 = tau * tau / 2.0;
    for (int j0 = 0; j0 < d.p; j0 += 4) {   // prop_full <- theta, loads ahead of the stores
        double t[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) if (j0 + q < d.p) t[q] = d.theta[(int64_t)(j0 + q) * C + c];
#pragma unroll
        for (int q = 0; q < 4; ++q) if (j0 + q < d.p) d.prop_full[(int64_t)(j0 + q) * C + c] = t[q];
    }
    if (d.rng_mode == EXTMCMC_RNG_REPLAY) {
        for (int i = 0; i < n; ++i)
            d.prop_full[(int64_t)u.coords_dev[i] * C + c] = d.rp_prop[((int64_t)sd.replay_row * d.p_u_max + i) * d.gC + d.g0 + c];
        d.n_used[c] = 0;
    } else {
        ChainStepStream rng(d.seed, (uint64_t)(d.chain_offset + c), sd.mcmciter, sd.pidx);
        for (int i = 0; i < n; i += 2) {
            const double u1 = rng.next(), u2 = rng.next();
            const double rad = sqrt(-2.0 * log(u1));
            double sn, cs;
            sincospi(2.0 * u2, &sn, &cs);
#pragma unroll
            for (int q = 0; q < 2; ++q) {
                if (i + q >= n) break;
                const int64_t j = u.coords_dev[i + q];
                const double th = d.theta[j * C + c];
                const double g = d.grad_cur[j * C + c] + mala_prior_grad<SP>(u, th, C, c, 0, i + q);
                d.prop_full[j * C + c] = th + h2 * g + tau * (rad * (q ? sn : cs));
            }
        }
        d.n_used[c] = rng.j;
    }
    law_prepare<SP>(d, c, d.prop_full + c, C);
}

// MALA accept/reject.  log q(a -> b) = -|b - a - (tau^2/2) g(a)|^2 / (2 tau^2) (the
// normalising constant is the same in both directions and is left out).
// The chain's own thread: decision, commit, history, counters; cs: staging (see CoopStage; with
// cs->m the covariance update is left to update_cov_coop).
// HANDOVER = false: the caller passes grad_prop / dsum_prop on to grad_cur / dsum_cur itself
// (mala_handover_coop: the rows are shared by the threads that have nothing else to do).
template <class SP = SpecAny, bool HANDOVER = true>
__device__ __forceinline__ Decision mala_decide_commit(const DevState &d, const StepDesc &sd, const DevUpdate &u, int64_t c) {
    const int64_t C = d.C;
    const int n = u.n_coords;
    const double tau = u.eps[c], h2 = tau * tau / 2.0;
    double qf = 0.0, qb = 0.0, lp_prop = 0.0, lp_cur = 0.0;
    for (int i0 = 0; i0 < n; i0 += 2) {   // loads of two coordinates in flight; sums in index order
        double a[2], b[2], ga[2], gb[2];
#pragma unroll
        for (int q = 0; q < 2; ++q)
            if (i0 + q < n) {
                const int64_t j = u.coords_dev[i0 + q];
                a[q] = d.theta[j * C + c];
                b[q] = d.prop_full[j * C + c];
                ga[q] = d.grad_cur[j * C + c];
                gb[q] = d.grad_prop[j * C + c];
            }
#pragma unroll
        for (int q = 0; q < 2; ++q)
            if (i0 + q < n) {
                const double gaq = ga[q] + mala_prior_grad<SP>(u, a[q], C, c, 0, i0 + q);
                const double gbq = gb[q] + mala_prior_grad<SP>(u, b[q], C, c, 1, i0 + q);
                const double rf = b[q] - a[q] - h2 * gaq, rb = a[q] - b[q] - h2 * gbq;
                qf += rf * rf;
                qb += rb * rb;
                if (SP::kLean || u.prior != EXTMCMC_PRIOR_USER) {
                    lp_prop += prior_logpdf1(u, b[q]);
                    lp_cur += prior_logpdf1(u, a[q]);
                }
            }
    }
    if (!SP::kLean && u.prior == EXTMCMC_PRIOR_USER) {   // the prior kernel's values (mala_prior_grad)
        lp_cur = u.prior_dev[c];
        lp_prop = u.prior_dev[(int64_t)(1 + n) * C + c];
    }
    const double inv = 1.0 / (2.0 * tau * tau);
    qf = -qf * inv;  // theta -> theta°
    qb = -qb * inv;  // theta° -> theta
    const double ll_prop = d.ll_prop[c];
    const double ll_cur = sd.first ? -INFINITY : d.ll[c];
    double llr = ll_prop - ll_cur;  // same association as run.jl:271-277
    llr = llr + qb;
    llr = llr - qf;
    llr = llr + lp_prop;
    llr = llr - lp_cur;
    const double E = draw_exp(d, sd, c);
    const bool accepted = E > -llr;
    const double ll_new = accepted ? ll_prop : ll_cur;
    if (accepted) {
        for (int i = 0; i < n; ++i) {
            const int64_t j = u.coords_dev[i];
            d.theta[j * C + c] = d.prop_full[j * C + c];
        }
        for (int j0 = 0; HANDOVER && j0 < d.p; j0 += 4) {   // grad_cur <- grad_prop
            double g[4];
#pragma unroll
            for (int q = 0; q < 4; ++q) if (j0 + q < d.p) g[q] = d.grad_prop[(int64_t)(j0 + q) * C + c];
#pragma unroll
            for (int q = 0; q < 4; ++q) if (j0 + q < d.p) d.grad_cur[(int64_t)(j0 + q) * C + c] = g[q];
        }
        if (HANDOVER && d.dsum_cur) {   // data-sum cache: the proposal's sums become the current state's
            const int rows = d.dsum_rows;
            for (int r0 = 0; r0 < rows; r0 += 4) {
                double g[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) if (r0 + q < rows) g[q] = d.dsum_prop[(int64_t)(r0 + q) * C + c];
#pragma unroll
                for (int q = 0; q < 4; ++q) if (r0 + q < rows) d.dsum_cur[(int64_t)(r0 + q) * C + c] = g[q];
            }
        }
    }
    return Decision{accepted, ll_new, ll_prop};
}
// What an accepted MALA proposal hands over to the current state -- the gradient and, with the data-sum
// cache, its sums: p + dsum_rows rows per chain, copied by the threads of slices [s0, s0 + ns) of an
// nch-chains-per-slice CTA (acc[ch] = the chain's decision, written before a CTA barrier).
__device__ __forceinline__ void mala_handover_coop(const DevState &d, int64_t c0, int nch, const uint8_t *acc,
                                                   int tid, int s0, int ns) {
    const int ch = tid % nch, slice = tid / nch - s0;
    const int64_t C = d.C, c = c0 + ch;
    if (slice < 0 || slice >= ns || c >= C || !acc[ch]) return;
    const int rows = d.p + (d.dsum_cur ? d.dsum_rows : 0);
#pragma unroll 2
    for (int r = slice; r < rows; r += ns) {
        if (r < d.p) d.grad_cur[(int64_t)r * C + c] = d.grad_prop[(int64_t)r * C + c];
        else d.dsum_cur[(int64_t)(r - d.p) * C + c] = d.dsum_prop[(int64_t)(r - d.p) * C + c];
    }
}
template <class SP = SpecAny>
__device__ __forceinline__ void mala_decide(const DevState &d, const StepDesc &sd, const DevUpdate &u, int64_t c,
                                            const CoopStage *cs) {
    const Decision dec = mala_decide_commit<SP>(d, sd, u, c);
    post_decision<SP>(d, sd, u, c, dec.accepted, dec.ll_new, dec.ll_prop, 1, cs);
}

}  // namespace extmcmc
