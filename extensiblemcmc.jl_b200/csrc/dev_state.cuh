// Device-resident chain state (SoA, chain fastest) and the per-step descriptor.
//
// Replaces the reference's host AoS-of-Vectors workspaces:
//   StandardGlobalSubworkspace   src/workspaces.jl:157-180  (state, histories)
//   StandardLocalSubworkspace    src/workspaces.jl:413-431  (local state, ll, ll_history)
//   GenericLocalWorkspace        src/workspaces.jl:453-458  (acceptance_history)
//   GenericChainStats            src/chain_statistics.jl:16-38
//   UniformRandomWalk.eps / AdaptationUnifRW counters
//                                src/transition_kernels/random_walk.jl:45-48,
//                                src/transition_kernels/adaptation.jl:51-61
#pragma once
#include <cstdint>
#include "../../include/extmcmc.h"

namespace extmcmc {

constexpr int kMaxCoords = 32;       // p_u limit of the random-walk updates (MALA: unlimited, coords_dev)
constexpr int kMaxPriorFactors = 16; // ProductPrior factors
constexpr int kMaxPriorParams = 1 + 4 * kMaxPriorFactors;
constexpr int kDataCacheMaxG = 16;   // most observation groups the data-sum cache serves (= kCoopG, step_kernels.cu)
constexpr int kMaxObsDim = 16;       // general-d Gaussian law on the device: d <= 16

// Laws whose sweep finishes ll (into ssum / ll_prop) and the gradient itself: the step kernels take
// the log-likelihood as it comes and prepare no law constants.
__host__ __device__ constexpr bool law_self_finished(int law) {
    return law == EXTMCMC_LAW_LOGISTIC || law == EXTMCMC_LAW_USER;
}

// prior families the compact (SpecLean) step kernels carry
inline bool lean_prior(int kind) {
    return kind == EXTMCMC_PRIOR_IMPROPER || kind == EXTMCMC_PRIOR_IMPROPER_POS || kind == EXTMCMC_PRIOR_NORMAL;
}

// One update as the kernels see it (constant per run; lives in a device table).
struct DevUpdate {
    int32_t kernel, n_coords, prior, adapt_kind;
    int32_t coords[kMaxCoords];
    uint8_t pos[kMaxCoords];
    double  prior_params[kMaxPriorParams];
    const double *prior_dev; // MVNORMAL prior: { mu[n], L[n*n] column-major lower Cholesky factor } (device)
    int32_t adapt_every_k;
    double  target, scale, vmin, vmax, offset;
    double *eps;          // [n_coords][C] per-chain step size (rw.eps, adapted in place)
    int32_t *adapt_prop;  // [C] AdaptationUnifRW.proposed
    int32_t *adapt_acc;   // [C] AdaptationUnifRW.accepted
    int64_t *tot_prop;    // [C] totals since set_state
    int64_t *tot_acc;     // [C]
    double  *ra_val;      // [C] latest rolling acceptance rate of this update
    uint8_t *acc_ring;    // [W][C] acceptance bits of the last W iterations
    // Gaussian random walks (random_walk.jl:123-232).  The Cholesky factors are cached: L_A once
    // per set_update (Sigma_A is shared by all chains and never changes), L_B per chain whenever
    // the Haario adaptation rewrites Sigma_B (L_B[0] = NaN marks "not positive definite").
    double *sigA;         // [n*n] column-major, shared by all chains (GaussianRandomWalk.Sigma / gsn_A)
    double *LA;           // [n*n] lower Cholesky factor of Symmetric(sigA) (upper triangle), column-major
    double *sigB;         // [n*n][C] per chain (gsn_B.Sigma, rewritten by the Haario adaptation)
    double *LB;           // [n*n][C] per chain factor of sigB
    double *hmean;        // [n][C]   HaarioTypeAdaptation.mean
    double *hcov;         // [n*n][C] HaarioTypeAdaptation.cov
    int32_t *coords_dev;  // [n_coords] device copy of coords (MALA: n_coords may exceed kMaxCoords)
};

// One schedule element (src/schedule.jl:56-66) plus what the host planner knows.
struct StepDesc {
    int64_t mcmciter;       // 1-based, enters compute_delta (adaptation.jl:312-319)
    int64_t seq;            // executed-step sequence number since set_state
    int64_t stat_n;         // GenericChainStats.N before this step (= seq + 1)
    int64_t xseq;           // executed-step sequence number since handle creation (never reset:
                            // parity and tag of the cross-rank exchange, go-flag of the block kernels)
    double  lambda;         // GaussianRandomWalkMix.lambda in force at this step (host-evaluated f_lambda)
    int32_t pidx;           // 0-based update index
    int32_t first;          // prev_pidx === nothing: ll stays -Inf (run.jl:76,109)
    int32_t ra_prev_valid;  // rolling_ar[max(1, iter-1)][pidx] was written (else 0.0)
    int32_t acc_out_valid;  // acceptance_history[iter - W] of this update was written
    int32_t replay_row;     // row of this step in the replay buffers
    int32_t haario_ready;   // this step brings the update's own-turn counter M to k (adaptation.jl:416-420)
    int32_t need_cur_grad;  // MALA: the gradient at the current state is stale (another update moved it)
    int32_t pad_;
};

struct DevState {
    int64_t C;              // chains on this rank (= the chain stride of every per-chain array below)
    int64_t chain_offset;   // global id of local chain 0
    // The persistent block kernels stage a CTA's own chains into shared memory and hand the
    // per-chain functions a VIEW of this struct (pointers into shared memory, C = chains of the CTA,
    // chain_offset moved).  Arrays that stay in global memory in such a view -- the history ring,
    // the replay buffers, the sweep partials -- keep the global chain stride gC and start at chain
    // g0; in the ordinary (global) state gC = C, g0 = 0.
    int64_t gC, g0;
    int64_t n_obs_total;    // N over all ranks (enters the log-likelihood constant)
    int32_t p, NU, W, H;    // params, updates, rolling window, history ring length
    int32_t law, stats_mode, rng_mode, p_u_max;
    int32_t n_haario;       // updates with HaarioTypeAdaptation (they register on every step)
    int32_t lean;           // host-side fact: every update set so far is a uniform random walk or MALA
                            // with an Improper / ImproperPos / Normal prior and no Haario adaptation ->
                            // the launchers pick the SpecLean instantiations (step_device.cuh)
    int32_t obs_dim, lawc_k;  // observation dimension; per-chain law constants in lawc
    int32_t G;              // observation groups (HIER_NORMAL; 1 otherwise)
    double *ll_prop;        // [C] finalized proposal log-likelihood (gradient path)
    double *grad_cur;       // [p][C] d ll / d theta at the current state
    double *grad_prop;      // [p][C] ... at the proposal
    // Data-sum cache (HIER_NORMAL, api.cu: data_cache_on): the per-group sums of both orders of the
    // CURRENT state and of the proposal in flight, laid out like a partial buffer with one segment per
    // group ([2][G][C]).  They depend on theta_1..G only, so an update of mu / tau reuses them instead
    // of streaming the observations again.  NULL: no cache.
    double *dsum_cur, *dsum_prop;
    uint64_t seed;
    // current state
    double *theta;          // [p][C]
    double *ll;             // [C] log-likelihood of the current state
    // proposal of the step in flight
    double *prop_loc;       // [kMaxCoords][C] local proposal theta°_loc
    double *prop_full;      // [p][C] full proposal = theta with coords replaced (run.jl:237-239)
    double *lawc;           // [lawc_k][C] per-chain law constants of the proposal
    uint32_t *n_used;       // [C] uniforms consumed by the proposal (next index = Exp draw)
    // per-chain scratch of the Gaussian walks / MvNormal priors / general-d law (SoA, so that a
    // thread-per-chain triangular solve stays coalesced and nothing lives in local memory)
    double *gw;             // [3 * gw_n][C]: z | t | m
    int32_t gw_n;
    double *mv_L;           // [d*d][C] Cholesky scratch of the general-d law
    // sweep output
    double *partial;        // [2][G*S][C] per-segment partial sums: q = 0 second-order, q = 1 first-order
    int32_t S;
    double *ssum;           // [C] reduced (and, under obs sharding, all-reduced) sums
    int32_t use_ssum;       // accept kernel reads ssum instead of partial
    // chain statistics
    double *mean;           // [p][C]
    double *cov;            // [p*p][C] (stats_mode 0) or [p][C] diagonal (stats_mode 1)
    // history ring, slot = seq % H
    double *h_theta;        // [H][p][C]
    double *h_prop;         // [H][p][C]
    double *h_ll;           // [H][C]
    double *h_llp;          // [H][C]
    uint8_t *h_acc;         // [H][C]
    // replay buffers (EXTMCMC_RNG_REPLAY)
    const double *rp_prop;  // [rows][p_u_max][C]
    const double *rp_exp;   // [rows][C]
    // fused cross-GPU exchange of the per-chain sums under observation sharding (no NCCL on the
    // hot path): every rank stores its sums into cell [parity][rank][chain] of every rank's rx
    // buffer over NVLink peer mappings; a cell is two 8-byte words that each carry the exchange's
    // sequence tag (exchange.cuh), so there is no fence and no flag; the consumer polls the cells and
    // adds them in rank order (identical totals on every rank).  parity = xseq & 1, tag = xseq + 1:
    // xseq is never reset, so a cell is only rewritten two exchanges later, after every rank has
    // consumed it.
    int32_t p2p, rank, world;
    unsigned long long **peer_rx;       // [world] -> rx[2][world][C][2] of each rank
    unsigned long long *my_rx;
    unsigned long long p2p_timeout_ns;  // bounded wait for the peers' cells
    int32_t *err_flag;      // sticky: 1 = a chain left the law's domain, 2 = peer exchange timed out
                            // (2: every later step is a no-op until the host has seen it)
    DevUpdate *upd;         // [NU]
};

}  // namespace extmcmc
