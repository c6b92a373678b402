// K1 (proposal), K3 (accept / commit / statistics / adaptation) and the MALA kernels of the
// per-step path: one kernel per stage of an update step -- the default path for every law, transition
// kernel and shape (the persistent block kernels of block_kernels.cu are opt-in variants).  Every
// kernel exists in a general instantiation (SpecAny) and in lean ones (SpecLean<LAW>, step_device.cuh)
// the host picks per handle.  One thread owns a chain's scalar work; the reductions of the sweep's
// partial sums and the covariance update of mid-sized models are shared by the 8 "slices" (threads) a
// CTA assigns to every chain, and the next element's proposal runs on the lanes of a second warp.  Compiled with -fmad=false: the
// reference never contracts a*b+c, and the replay parity tests compare eps, running moments and
// trajectories bit-for-bit against the CPU oracle.
#include <cmath>
#include <cstdint>
#include <cuda_runtime.h>
#include "dev_state.cuh"
#include "philox.cuh"
#include "step_device.cuh"
#include "step_kernels.h"
#include "tma.cuh"
#include "exchange.cuh"
#include "sweep.h"

namespace extmcmc {

// a peer exchange timed out earlier: nothing is committed any more until the host has seen it
__device__ __forceinline__ bool exchange_failed(const DevState &d) {
    return *reinterpret_cast<volatile int32_t *>(d.err_flag) == 2;
}

// ---------------------------------------------------------------------------------
// K1: proposal!  (step_device.cuh: propose_chain)
// ---------------------------------------------------------------------------------
template <class SP>
__global__ void __launch_bounds__(256)
propose_kernel(DevState d, const StepDesc *__restrict__ descs, int k) {
    __shared__ StepCtx ctx;
    load_step_ctx(&ctx, d, descs, k, threadIdx.x, blockDim.x, CtaSync{});
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C || exchange_failed(d)) return;
    propose_chain<SP>(d, ctx.sd, ctx.u, c);
}

// Law constants of the CURRENT state (extmcmc_eval_loglik).
__global__ void __launch_bounds__(256) prepare_current_kernel(DevState d) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    law_prepare(d, c, d.theta + c, d.C);
}

// Cholesky factor of a Sigma shared by all chains (GaussianRandomWalk.Sigma / gsn_A), or of the
// initial per-chain Sigma_B of every chain: one thread per matrix.
__global__ void chol_factor_kernel(double *S, double *L, int n, int64_t stride, int64_t count) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= count) return;
    chol_lower_sym_upper(MatRef{S + c, stride}, n, MatRef{L + c, stride});
}

constexpr int kRedThreads = 256;

template <int kRedSlices>
__device__ __forceinline__ double reduce_segments(const DevState &d, double *sh /*[SL][256/SL]*/) {
    constexpr int kRedChains = kRedThreads / kRedSlices;
    const int lane_c = threadIdx.x % kRedChains;
    const int slice = threadIdx.x / kRedChains;
    const int64_t c = (int64_t)blockIdx.x * kRedChains + lane_c;
    double s = 0.0;
    if (c < d.C) {
        const double *p = d.partial + c;
        const int nrows = d.S * d.G;   // all segments of all observation groups
        // all loads of a batch are issued before the first add (memory-level parallelism: after a
        // large sweep these come from DRAM); the adds stay in increasing row order
        int i = slice;
        for (; i + 7 * kRedSlices < nrows; i += 8 * kRedSlices) {
            double a[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) a[q] = p[(int64_t)(i + q * kRedSlices) * d.C];
#pragma unroll
            for (int q = 0; q < 8; ++q) s += a[q];
        }
        for (; i < nrows; i += kRedSlices) s += p[(int64_t)i * d.C];
    }
    if (kRedSlices == 1) return s;
    sh[slice * kRedChains + lane_c] = s;
    __syncthreads();
    double tot = 0.0;
    if (slice == 0) {
#pragma unroll
        for (int j = 0; j < kRedSlices; ++j) tot += sh[j * kRedChains + lane_c];
    }
    return tot;  // valid in threads with slice == 0
}

// Per-group sums of both orders, out[q][g][c] = sum_i partial[q][g*S + i][c] (segment order): what a
// rank contributes to the all-reduce of a gradient sweep under observation sharding.  The MALA
// kernels then read `out` as a partial buffer with one segment per group.
__global__ void __launch_bounds__(256) reduce_group_sums_kernel(DevState d, double *__restrict__ out) {
    const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t C = d.C;
    if (idx >= (int64_t)2 * d.G * C) return;
    const int64_t r = idx / C, c = idx % C;          // r = q * G + g
    const double *p = d.partial + (r * d.S) * C + c;  // rows (q G + g) S .. + S of partial[2][G S][C]
    double s = 0.0;
    int i = 0;
    for (; i + 3 < d.S; i += 4) {
        double a[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) a[q] = p[(int64_t)(i + q) * C];
#pragma unroll
        for (int q = 0; q < 4; ++q) s += a[q];
    }
    for (; i < d.S; ++i) s += p[(int64_t)i * C];
    out[idx] = s;
}

template <int SL>
__global__ void __launch_bounds__(256) reduce_partials_kernel(DevState d) {
    __shared__ double sh[kRedThreads];
    constexpr int kRedChains = kRedThreads / SL;
    const double tot = reduce_segments<SL>(d, sh);
    const int64_t c = (int64_t)blockIdx.x * kRedChains + (threadIdx.x % kRedChains);
    if ((threadIdx.x / kRedChains) == 0 && c < d.C) d.ssum[c] = tot;
}

// Reduce this rank's partial sums and push them to every rank (itself included) through peer
// pointers, as tagged cells (exchange.cuh): nothing else to signal.
template <int SL>
__global__ void __launch_bounds__(256)
reduce_push_kernel(DevState d, const StepDesc *__restrict__ descs, int k) {
    __shared__ double sh[kRedThreads];
    constexpr int kRedChains = kRedThreads / SL;
    // PDL chain sweep -> reduce_push -> accept: start early, let the accept kernel start early
    // too (its prologue then overlaps the sweep), and wait for the sweep before touching its sums
    griddep_launch_dependents();
    const StepDesc sd = descs[k];
    const int parity = (int)(sd.xseq & 1);
    griddep_wait();
    const double tot = reduce_segments<SL>(d, sh);
    const int64_t c = (int64_t)blockIdx.x * kRedChains + (threadIdx.x % kRedChains);
    if ((threadIdx.x / kRedChains) == 0 && c < d.C) {
        const int64_t cell = ll_cell(parity, d.world, d.rank, d.C, c);
        const uint32_t tag = (uint32_t)(sd.xseq + 1);
        for (int q = 0; q < d.world; ++q) ll_store(d.peer_rx[q] + cell, tot, tag);
    }
}

// Wait until every rank's sums of this step have landed, then add them in rank order.  ok = false
// (CTA-uniform) when the wait timed out: the caller must not commit anything.
// `reader`: the threads that need the sum (one per chain).
__device__ __forceinline__ double wait_and_combine(const DevState &d, const StepDesc &sd, int64_t c, bool reader, bool &ok) {
    const int parity = (int)(sd.xseq & 1);
    const uint32_t tag = (uint32_t)(sd.xseq + 1);
    double s = 0.0;
    int mine = 1;
    if (reader && c < d.C) {
        const unsigned long long t0 = global_timer_ns();
        for (int r = 0; r < d.world && mine; ++r) {
            double v;
            if (ll_load(d.my_rx + ll_cell(parity, d.world, r, d.C, c), tag, v, t0, d.p2p_timeout_ns)) s += v;
            else { atomicExch(d.err_flag, 2); mine = 0; }
        }
    }
    ok = __syncthreads_and(mine) != 0;
    return s;
}

__global__ void __launch_bounds__(256) finalize_loglik_kernel(DevState d, double *ll_out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    ll_out[c] = law_finalize(d, c, d.ssum[c], d.theta + c);
}

// ---------------------------------------------------------------------------------
// Deferred bookkeeping.  What feeds the next sweep is the decision, the commit and the next proposal;
// running moments, rolling acceptance rate, totals and adaptation of a step feed nothing before the
// SAME update's next turn.  In the lean, sliced instantiations the kernel that decides step k - 1
// therefore writes only the history row and leaves the rest to the first step kernel of step k, which
// runs it in its prologue -- resident through PDL while the sweep of step k is still streaming -- on
// warps of its own: moments on the chains' lanes of warp 3, counters on those of warp 2, then the
// cooperative covariance update by all threads.  Both sides evaluate the same predicate: the host says
// whether a producer / consumer exists (flags, from the block's kernel kinds), the device checks that
// the two elements name different updates (the next proposal of the same update must see its adapted
// step size, so that case stays in place).  The last element of a block is never deferred.
// ---------------------------------------------------------------------------------
constexpr int kFlagConsume = 1, kFlagDefer = 2;
// kFlagNoSweep: no likelihood sweep precedes this step kernel (data-sum cache, dev_state.cuh): its
// stream predecessor is the step kernel of the previous element, whose writes it must wait for
// before it reads anything but the descriptors.
constexpr int kFlagNoSweep = 4;

template <class SP>
__device__ __forceinline__ void run_deferred(const DevState &d, const StepCtx &prev, int64_t c0, int nch, bool stage,
                                             double *sh_t, double *sh_m, double *sh_n) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    const int64_t c = c0 + (tid % nch);
    const bool lane_ok = lane < nch && c < d.C;
    const bool coop = stage && d.stats_mode == 0;   // CTA-uniform
    const CoopStage cs{sh_t, coop ? sh_m : nullptr, sh_n, nch, tid % nch};
    // moments: per-parameter work only (cooperative covariance, variances or no statistics) is shared by
    // warps 3.. in groups of four parameters; the thread-alone full covariance stays on warp 3
    const bool multi = coop || d.stats_mode != 0;   // CTA-uniform
    const int nw = (int)(blockDim.x >> 5);
    if (w >= 3 && lane_ok && (multi || w == 3)) {
        post_decision_moments<SP, false, true>(d, prev.sd, c, false, 0.0, 0.0, stage ? &cs : nullptr,
                                               multi ? w - 3 : 0, multi ? nw - 3 : 1);
    } else if (w == 2 && lane_ok) {
        const bool acc = d.h_acc[(prev.sd.seq % d.H) * d.gC + d.g0 + c] != 0;
        const int n_eps = prev.u.kernel == EXTMCMC_KERNEL_MALA ? 1 : prev.u.n_coords;   // lean: uniform walk or MALA
        post_decision_counters<SP>(d, prev.sd, prev.u, c, acc, n_eps);
    }
    if (coop) {
        __syncthreads();
        update_cov_coop(d, prev.sd.stat_n, c0, nch, sh_t, sh_m, sh_n, tid, blockDim.x);
    }
    // the deferred work has read the state of step k - 1 (and the staging): only now may this step commit
    __syncthreads();
}

// ---------------------------------------------------------------------------------
// K3: accept_reject! (src/run.jl:268-281) for the random-walk updates.
// ---------------------------------------------------------------------------------
template <int SL, class SP>
__global__ void __launch_bounds__(256)
accept_kernel(DevState d, const StepDesc *__restrict__ descs, int k, int fuse_next, int flags) {
    // 256 threads = (256/SL) chains x SL reduction slices; slice 0 carries on with the chain
    constexpr int kRedChains = kRedThreads / SL;
    __shared__ double sh[kRedThreads];
    __shared__ StepCtx ctx, ctx_next, ctx_prev;
    // staging of the cooperative covariance update (only the sliced layouts have spare threads)
    constexpr int kStage = SL >= 8 ? kCoopP * kRedChains : 1;
    __shared__ double sh_t[kStage], sh_m[kStage], sh_n[kStage];
    // PDL: this kernel may have been scheduled while the likelihood sweep is still running.
    // Everything up to griddep_wait() only READS state that was final before the sweep started
    // (chain state, proposal, step sizes, law constants, RNG counters) -- the transition-density
    // and prior terms and the Exp(1) draw are computed here, hidden behind the sweep.
    griddep_launch_dependents();
    constexpr bool kCanDefer = SL >= 8 && SP::kLean;
    const bool may_defer = kCanDefer && (flags & kFlagDefer), may_consume = kCanDefer && (flags & kFlagConsume);
    load_step_ctx(&ctx, d, descs, k, threadIdx.x, blockDim.x, CtaSync{});
    if (fuse_next == 1 || may_defer) load_step_ctx(&ctx_next, d, descs, k + 1, threadIdx.x, blockDim.x, CtaSync{});
    if (may_consume) load_step_ctx(&ctx_prev, d, descs, k - 1, threadIdx.x, blockDim.x, CtaSync{});
    const int64_t c = (int64_t)blockIdx.x * kRedChains + (threadIdx.x % kRedChains);
    if (flags & kFlagNoSweep) griddep_wait();   // the predecessor is a step kernel, not a sweep
    const bool dead = exchange_failed(d);   // CTA-uniform
    const bool worker = (threadIdx.x / kRedChains) == 0 && c < d.C && !dead;
    const StepDesc &sd = ctx.sd;
    const DevUpdate &u = ctx.u;
    // full covariance of a model with more than a handful of parameters: all slices share the work
    const bool stage = SL >= 8 && d.p > 4 && d.p <= kCoopP;   // CTA-uniform
    const bool coop = stage && d.stats_mode == 0;
    RwPre pre{};
    if (worker) pre = rw_accept_prologue<SP>(d, sd, u, c);
    // bookkeeping the previous element left to us (other warps; the worker lanes join when they are done)
    if (may_consume && !dead && ctx_prev.sd.pidx != sd.pidx)
        run_deferred<SP>(d, ctx_prev, (int64_t)blockIdx.x * kRedChains, kRedChains, stage, sh_t, sh_m, sh_n);

    griddep_wait();   // the sweep (and, under sharding, the exchange) has finished
    if (dead) return;
    double S;
    if (d.p2p) {
        bool ok;
        S = wait_and_combine(d, ctx.sd, c, (threadIdx.x / kRedChains) == 0 && !dead, ok);
        if (!ok) return;   // nothing is committed; the sticky flag turns the steps to come into no-ops
    } else if (d.use_ssum) {
        S = c < d.C ? d.ssum[c] : 0.0;
    } else {
        S = reduce_segments<SL>(d, sh);
    }
    const CoopStage cs{sh_t, coop ? sh_m : nullptr, sh_n, kRedChains, (int)(threadIdx.x % kRedChains)};
    // Task split (lean instantiations, sliced layouts): once the decision is committed, the next
    // element's proposal runs on the chains' lanes of warp 1 while the worker lanes (warp 0) do the
    // bookkeeping -- both are latency-bound single-warp instruction streams.  Not when the next
    // element is the same update: its proposal must see this step's adapted step size.
    const bool split = SL >= 8 && SP::kLean && fuse_next == 1 && ctx_next.sd.pidx != sd.pidx;   // CTA-uniform
    const bool defer = may_defer && ctx_next.sd.pidx != sd.pidx;                                  // CTA-uniform
    if (defer) {
        // only what the next sweep and the history need: decision, commit, history row, next proposal
        const bool prop_lane = fuse_next == 1 && (threadIdx.x >> 5) == 1 && (threadIdx.x & 31) < kRedChains && c < d.C;
        Decision dec{};
        if (worker) dec = rw_decide_commit<SP>(d, u, c, pre, S);
        __syncthreads();   // the committed state is visible to the proposal lanes and to the history lanes
        // history row: the chain's thread writes the scalars and the first four parameters, the chains'
        // lanes of warps 2.. the other groups of four
        const int wv = threadIdx.x >> 5, n_grp = (int)(blockDim.x >> 5) - 1;
        const bool hist_lane = wv >= 2 && (threadIdx.x & 31) < kRedChains && c < d.C;
        if (worker) post_decision_moments<SP, true, false>(d, sd, c, dec.accepted, dec.ll_new, dec.ll_prop, nullptr, 0, n_grp);
        else if (prop_lane) propose_draw<SP>(d, ctx_next.sd, ctx_next.u, c);
        else if (hist_lane) post_decision_moments<SP, true, false>(d, sd, c, false, 0.0, 0.0, nullptr, wv - 1, n_grp);
        if (fuse_next == 1) {
            __syncthreads();   // prop_full has been read for the history row
            if (prop_lane) propose_set<SP>(d, ctx_next.u, c);
        } else if (fuse_next == 2 && worker) {
            law_prepare<SP>(d, c, d.theta + c, d.C);
        }
        return;
    }
    if (split) {
        // lanes of warp 1: the next proposal; lanes of warp 2: rolling acceptance rate, totals, adaptation
        const bool lane_ok = (threadIdx.x & 31) < kRedChains && c < d.C;
        const bool prop_lane = (threadIdx.x >> 5) == 1 && lane_ok;
        const bool cnt_lane = (threadIdx.x >> 5) == 2 && lane_ok;
        __shared__ uint8_t sh_acc[kRedChains];
        Decision dec{};
        if (worker) {
            dec = rw_decide_commit<SP>(d, u, c, pre, S);
            sh_acc[threadIdx.x % kRedChains] = dec.accepted ? 1 : 0;
        }
        __syncthreads();   // the committed state and the decisions are visible to the other warps
        if (worker) post_decision_moments<SP>(d, sd, c, dec.accepted, dec.ll_new, dec.ll_prop, stage ? &cs : nullptr);
        else if (prop_lane) propose_draw<SP>(d, ctx_next.sd, ctx_next.u, c);
        else if (cnt_lane) post_decision_counters<SP>(d, sd, u, c, sh_acc[threadIdx.x % kRedChains] != 0, rw_n_eps<SP>(u));
        __syncthreads();   // prop_full has been read for the history row; the staging is complete
        if (prop_lane) propose_set<SP>(d, ctx_next.u, c);
        if (coop)
            update_cov_coop(d, sd.stat_n, (int64_t)blockIdx.x * kRedChains, kRedChains, sh_t, sh_m, sh_n, threadIdx.x, blockDim.x);
        return;
    }
    if (worker) rw_accept_finish<SP>(d, sd, u, c, pre, S, stage ? &cs : nullptr);
    if (coop) {
        __syncthreads();
        update_cov_coop(d, sd.stat_n, (int64_t)blockIdx.x * kRedChains, kRedChains, sh_t, sh_m, sh_n, threadIdx.x, blockDim.x);
    }
    if (!worker) return;
    // proposal of the NEXT schedule element of this block, fused here: the chain's thread has just
    // committed its state, and one launch per update step is saved
    if (fuse_next == 2) law_prepare<SP>(d, c, d.theta + c, d.C);   // what prepare_current_kernel would do
    else if (fuse_next) propose_chain<SP>(d, ctx_next.sd, ctx_next.u, c);
}

// The MALA step kernels run as CTAs of kMalaChains chains x kMalaSlices slices (256 threads): the
// slices share the per-group segment sums of the hierarchical law and the covariance update, the
// chain's own thread (slice 0) does the scalar work.  Same sums, same order as grad_finalize_chain.
constexpr int kMalaChains = 32, kMalaSlices = 8;
constexpr int kCoopG = 16;   // most observation groups reduced this way
static_assert(kCoopG == kDataCacheMaxG, "the data-sum cache is filled by grad_finalize_coop");
template <class SP>
__device__ __forceinline__ void grad_finalize_coop(const DevState &d, int64_t c0, const double *__restrict__ src,
                                                   double *__restrict__ ll_out, double *__restrict__ grad_out,
                                                   double *sh2, double *sh1 /*[kCoopG][kMalaChains] each*/,
                                                   double *__restrict__ dsum_out = nullptr /*[2][G][C] or NULL*/) {
    const int ch = threadIdx.x % kMalaChains, slice = threadIdx.x / kMalaChains;
    const int64_t c = c0 + ch, C = d.C;
    const int G = d.G, S = d.S;
    if (sp_law<SP>(d) != EXTMCMC_LAW_HIER_NORMAL || G > kCoopG) {   // CTA-uniform
        if (slice == 0 && c < C) grad_finalize_chain<SP>(d, c, src, ll_out, grad_out);
        return;
    }
    const int64_t rows = (int64_t)G * S;
    if (c < C)
        for (int g = slice; g < G; g += kMalaSlices) {
            const double *p2 = d.partial + ((int64_t)g * S) * C + c;
            const double *p1 = d.partial + (rows + (int64_t)g * S) * C + c;
            double s2 = 0.0, s1 = 0.0;
            int i = 0;
            for (; i + 3 < S; i += 4) {   // loads first, adds in segment order
                double a[4], b[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) { a[q] = p2[(int64_t)(i + q) * C]; b[q] = p1[(int64_t)(i + q) * C]; }
#pragma unroll
                for (int q = 0; q < 4; ++q) { s2 += a[q]; s1 += b[q]; }
            }
            for (; i < S; ++i) { s2 += p2[(int64_t)i * C]; s1 += p1[(int64_t)i * C]; }
            sh2[g * kMalaChains + ch] = s2;
            sh1[g * kMalaChains + ch] = s1;
            if (dsum_out) { dsum_out[(int64_t)g * C + c] = s2; dsum_out[((int64_t)G + g) * C + c] = s1; }
        }
    __syncthreads();
    if (slice != 0 || c >= C) return;
    const double mu = src[(int64_t)G * C + c], tau = src[(int64_t)(G + 1) * C + c];
    if (!(tau > 0.0) || isinf(tau)) *d.err_flag = 1;   // the current state never went through law_prepare
    const double it2 = 1.0 / (tau * tau);
    double s2_tot = 0.0, dmu = 0.0, dev2 = 0.0;
    for (int g = 0; g < G; ++g) {
        s2_tot += sh2[g * kMalaChains + ch];
        const double dv = src[(int64_t)g * C + c] - mu;
        grad_out[(int64_t)g * C + c] = sh1[g * kMalaChains + ch] - dv * it2;
        dmu += dv * it2;
        dev2 += dv * dv;
    }
    grad_out[(int64_t)G * C + c] = dmu;
    grad_out[(int64_t)(G + 1) * C + c] = -(double)G / tau + dev2 * it2 / tau;
    ll_out[c] = law_finalize<SP>(d, c, s2_tot, src + c);
}

__global__ void __launch_bounds__(128)
grad_finalize_kernel(DevState d, const double *__restrict__ src, double *__restrict__ ll_out,
                     double *__restrict__ grad_out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    grad_finalize_chain(d, c, src, ll_out, grad_out);
}

// K5a: MALA proposal (step_device.cuh: mala_propose_chain)
template <class SP>
__global__ void __launch_bounds__(kMalaChains * kMalaSlices)
mala_propose_kernel(DevState d, const StepDesc *__restrict__ descs, int k, int finalize_cur,
                    double *__restrict__ ll_scratch, int flags) {
    __shared__ StepCtx ctx, ctx_prev;
    __shared__ double sh2[kCoopG * kMalaChains], sh1[kCoopG * kMalaChains];
    __shared__ double sh_t[kCoopP * kMalaChains], sh_m[kCoopP * kMalaChains], sh_n[kCoopP * kMalaChains];
    // PDL (as in accept_kernel): the schedule element and update entry are staged while the
    // preceding sweep is still running; nothing the predecessor writes is read before the wait
    griddep_launch_dependents();
    load_step_ctx(&ctx, d, descs, k, threadIdx.x, blockDim.x, CtaSync{});
    const int64_t c0 = (int64_t)blockIdx.x * kMalaChains;
    const int64_t c = c0 + threadIdx.x % kMalaChains;
    // bookkeeping the previous element left to us (see run_deferred).  Behind the current-state gradient
    // sweep when there is one (that sweep started after the previous step kernel had finished); otherwise
    // our predecessor IS that step kernel and we must wait for it first.
    const bool may_consume = SP::kLean && (flags & kFlagConsume);
    if (may_consume) load_step_ctx(&ctx_prev, d, descs, k - 1, threadIdx.x, blockDim.x, CtaSync{});
    const bool consume = may_consume && ctx_prev.sd.pidx != ctx.sd.pidx;
    // finalize_cur: 1 = a sweep of the current state precedes this kernel; 2 = its sums come from the
    // data-sum cache (d.partial is the cache, one segment per group): no sweep, the predecessor is a
    // step kernel like with 0
    const bool behind_sweep = finalize_cur == 1;
    if (consume && behind_sweep) run_deferred<SP>(d, ctx_prev, c0, kMalaChains, d.p <= kCoopP, sh_t, sh_m, sh_n);
    griddep_wait();
    if (consume && !behind_sweep) run_deferred<SP>(d, ctx_prev, c0, kMalaChains, d.p <= kCoopP, sh_t, sh_m, sh_n);
    // the sweep just before this kernel evaluated the CURRENT state: finish its sums here
    // (gradient of the current state) instead of in a kernel of its own
    if (finalize_cur)
        grad_finalize_coop<SP>(d, c0, d.theta, ll_scratch, d.grad_cur, sh2, sh1, behind_sweep ? d.dsum_cur : nullptr);
    if (SP::kLean && d.rng_mode != EXTMCMC_RNG_REPLAY) {   // CTA-uniform
        // The Box-Muller pairs of a chain's proposal are independent (counter-based stream: pair q
        // reads Philox block q): slice q % 8 draws pair q while the slices also share the copy of the
        // state into prop_full.  Same expressions as mala_propose_chain, coordinate by coordinate.
        if (finalize_cur) __syncthreads();   // grad_cur of this CTA's chains is complete
        const int slice = threadIdx.x / kMalaChains;
        const DevUpdate &u = ctx.u;
        const StepDesc &sd = ctx.sd;
        const int n = u.n_coords;
        const int64_t C = d.C;
        const bool live = c < C;
        if (live)
            for (int j = slice; j < d.p; j += kMalaSlices) d.prop_full[(int64_t)j * C + c] = d.theta[(int64_t)j * C + c];
        __syncthreads();   // the copy of the state is complete: the update's coordinates may be overwritten
        const double tau = live ? u.eps[c] : 1.0, h2 = tau * tau / 2.0;
        const int n_pairs = (n + 1) / 2;
        if (live)
            for (int q = slice; q < n_pairs; q += kMalaSlices) {
                ChainStepStream rng(d.seed, (uint64_t)(d.chain_offset + c), sd.mcmciter, sd.pidx, (uint32_t)(2 * q));
                const double u1 = rng.next(), u2 = rng.next();
                const double rad = sqrt(-2.0 * log(u1));
                double sn, cs;
                sincospi(2.0 * u2, &sn, &cs);
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    const int i = 2 * q + e;
                    if (i >= n) break;
                    const int64_t j = u.coords_dev[i];
                    const double th = d.theta[j * C + c];
                    const double g = d.grad_cur[j * C + c] + prior_grad(u, th);
                    d.prop_full[j * C + c] = th + h2 * g + tau * (rad * (e ? sn : cs));
                }
            }
        __syncthreads();
        if (slice != 0 || !live) return;
        d.n_used[c] = (uint32_t)(2 * n_pairs);
        law_prepare<SP>(d, c, d.prop_full + c, C);
        return;
    }
    if (threadIdx.x >= kMalaChains || c >= d.C) return;
    mala_propose_chain<SP>(d, ctx.sd, ctx.u, c);
}

// K5b: MALA accept/reject (step_device.cuh: mala_decide)
template <class SP>
__global__ void __launch_bounds__(kMalaChains * kMalaSlices)
mala_accept_kernel(DevState d, const StepDesc *__restrict__ descs, int k, int finalize_prop, int fuse_next, int flags) {
    __shared__ StepCtx ctx, ctx_next;
    __shared__ double sh2[kCoopG * kMalaChains], sh1[kCoopG * kMalaChains];
    __shared__ double sh_t[kCoopP * kMalaChains], sh_m[kCoopP * kMalaChains], sh_n[kCoopP * kMalaChains];
    griddep_launch_dependents();
    const bool may_defer = SP::kLean && (flags & kFlagDefer);
    load_step_ctx(&ctx, d, descs, k, threadIdx.x, blockDim.x, CtaSync{});
    if (fuse_next || may_defer) load_step_ctx(&ctx_next, d, descs, k + 1, threadIdx.x, blockDim.x, CtaSync{});
    griddep_wait();   // the gradient sweep of the proposal has finished
    const int64_t c0 = (int64_t)blockIdx.x * kMalaChains;
    const int ch = threadIdx.x % kMalaChains;
    const int64_t c = c0 + ch;
    if (finalize_prop) grad_finalize_coop<SP>(d, c0, d.prop_full, d.ll_prop, d.grad_prop, sh2, sh1, d.dsum_prop);
    const bool worker = threadIdx.x < kMalaChains && c < d.C;
    const bool stage = d.p <= kCoopP;   // CTA-uniform
    const bool coop = stage && d.stats_mode == 0;
    const CoopStage cs{sh_t, coop ? sh_m : nullptr, sh_n, kMalaChains, ch};
    // the decisions, for the threads that hand the proposal's gradient and data sums over (slices 3..7:
    // warps with no other task, next to the worker's bookkeeping and the next proposal)
    __shared__ uint8_t sh_acc[kMalaChains];
    if (may_defer && ctx_next.sd.pidx != ctx.sd.pidx) {   // deferred bookkeeping (see run_deferred)
        const bool prop_lane = fuse_next && (threadIdx.x >> 5) == 1 && c < d.C;
        Decision dec{};
        if (worker) {
            dec = mala_decide_commit<SP, false>(d, ctx.sd, ctx.u, c);
            sh_acc[ch] = dec.accepted ? 1 : 0;
        }
        __syncthreads();
        const int wv = threadIdx.x >> 5;
        if (worker) post_decision_moments<SP, true, false>(d, ctx.sd, c, dec.accepted, dec.ll_new, dec.ll_prop, nullptr, 0, kMalaSlices - 1);
        else if (prop_lane) propose_draw<SP>(d, ctx_next.sd, ctx_next.u, c);
        else {
            if (wv >= 2 && c < d.C)   // history row: groups of four parameters on the lanes of warps 2..
                post_decision_moments<SP, true, false>(d, ctx.sd, c, false, 0.0, 0.0, nullptr, wv - 1, kMalaSlices - 1);
            mala_handover_coop(d, c0, kMalaChains, sh_acc, threadIdx.x, 3, kMalaSlices - 3);
        }
        if (fuse_next) {
            __syncthreads();
            if (prop_lane) propose_set<SP>(d, ctx_next.u, c);
        }
        return;
    }
    if (SP::kLean && fuse_next) {   // task split as in accept_kernel (the next element is another update)
        const bool prop_lane = (threadIdx.x >> 5) == 1 && c < d.C;
        const bool cnt_lane = (threadIdx.x >> 5) == 2 && c < d.C;
        Decision dec{};
        if (worker) {
            dec = mala_decide_commit<SP, false>(d, ctx.sd, ctx.u, c);
            sh_acc[ch] = dec.accepted ? 1 : 0;
        }
        __syncthreads();
        if (worker) post_decision_moments<SP>(d, ctx.sd, c, dec.accepted, dec.ll_new, dec.ll_prop, stage ? &cs : nullptr);
        else if (prop_lane) propose_draw<SP>(d, ctx_next.sd, ctx_next.u, c);
        else if (cnt_lane) post_decision_counters<SP>(d, ctx.sd, ctx.u, c, sh_acc[ch] != 0, 1);
        else mala_handover_coop(d, c0, kMalaChains, sh_acc, threadIdx.x, 3, kMalaSlices - 3);
        __syncthreads();
        if (prop_lane) propose_set<SP>(d, ctx_next.u, c);
        if (coop) update_cov_coop(d, ctx.sd.stat_n, c0, kMalaChains, sh_t, sh_m, sh_n, threadIdx.x, blockDim.x);
        return;
    }
    if (worker) mala_decide<SP>(d, ctx.sd, ctx.u, c, stage ? &cs : nullptr);
    if (coop) {
        __syncthreads();
        update_cov_coop(d, ctx.sd.stat_n, c0, kMalaChains, sh_t, sh_m, sh_n, threadIdx.x, blockDim.x);
    }
    // next element is a random-walk update: issue its proposal here (one launch saved)
    if (worker && fuse_next) propose_chain<SP>(d, ctx_next.sd, ctx_next.u, c);
}

// ---------------------------------------------------------------------------------
// utilities
// ---------------------------------------------------------------------------------
// x_i ~ N(mean, sd^2), i = global observation index; Box-Muller on the Philox stream
// keyed by (seed; counter = i/2).  BASELINE cfg 5 generates 1e9 observations in place.
__global__ void generate_obs_normal_kernel(double *obs, int64_t first, int64_t n, double mean,
                                           double sd, uint64_t seed) {
    const int64_t pair0 = first >> 1;
    const int64_t n_pairs = ((first + n + 1) >> 1) - pair0;
    for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q < n_pairs;
         q += (int64_t)gridDim.x * blockDim.x) {
        const uint64_t pair = (uint64_t)(pair0 + q);
        const Philox4 w = philox4x32_10((uint32_t)pair, (uint32_t)(pair >> 32), 0x0B5E0B5Eu, 0u,
                                        (uint32_t)seed, (uint32_t)(seed >> 32));
        const double u1 = u52_to_unit(w.w[0], w.w[1]), u2 = u52_to_unit(w.w[2], w.w[3]);
        const double rad = sqrt(-2.0 * log(u1));
        double sn, cs;
        sincospi(2.0 * u2, &sn, &cs);
        const int64_t i0 = (int64_t)(pair << 1), i1 = i0 + 1;
        if (i0 >= first && i0 < first + n) obs[i0 - first] = mean + sd * (rad * cs);
        if (i1 >= first && i1 < first + n) obs[i1 - first] = mean + sd * (rad * sn);
    }
}

__global__ void flush_l2_kernel(double *buf, int64_t n, double v) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (int64_t)gridDim.x * blockDim.x)
        buf[i] = v;
}

// Dependent-free FP64 FMA chains: 16 accumulators per thread, the loop body unrolled 8 times
// (128 DFMA per 3 loop-control instructions), `iters` counts single FMA rounds over the 16.
__global__ void fp64_peak_kernel(double *out, int iters, double a, double b) {
    double acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = (double)(threadIdx.x + i);
#pragma unroll 1
    for (int it = 0; it < iters; it += 8) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
#pragma unroll
            for (int i = 0; i < 16; ++i) acc[i] = fma(acc[i], a, b);
        }
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 16; ++i) s += acc[i];
    if (s == 123.456) out[0] = s;
}

// Independent FP64 tensor-core MMA chains (mma.sync.m8n8k4.f64 -> SASS DMMA.8x8x4): 8 accumulator
// pairs per warp, 512 flop per instruction.
__global__ void dmma_peak_kernel(double *out, int iters, double a, double b) {
    double c[8][2];
#pragma unroll
    for (int i = 0; i < 8; ++i) { c[i][0] = (double)threadIdx.x; c[i][1] = (double)i; }
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < 8; ++i)
            asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                         : "+d"(c[i][0]), "+d"(c[i][1])
                         : "d"(a), "d"(b));
    }
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < 8; ++i) s += c[i][0] + c[i][1];
    if (s == 123.456) out[0] = s;
}

// ---------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------
static inline int blocks_for(int64_t C) { return (int)((C + 255) / 256); }

// Which instantiation serves this handle: the lean ones when the host found every update to be a
// uniform random walk or MALA with Improper / ImproperPos / Normal priors and no Haario adaptation
// (DevState.lean), per law; the general one otherwise.  F is called with a StepSpec value.
template <class F>
static inline void with_spec(const DevState &d, F f) {
    if (d.lean && d.law == EXTMCMC_LAW_GSN_IID_1D) f(SpecLean<EXTMCMC_LAW_GSN_IID_1D>{});
    else if (d.lean && d.law == EXTMCMC_LAW_HIER_NORMAL) f(SpecLean<EXTMCMC_LAW_HIER_NORMAL>{});
    else if (d.lean && law_self_finished(d.law)) f(SpecLean<EXTMCMC_LAW_LOGISTIC>{});
    else f(SpecAny{});
}
void launch_propose(const DevState &d, const StepDesc *descs, int k, cudaStream_t st) {
    with_spec(d, [&](auto sp) { propose_kernel<decltype(sp)><<<blocks_for(d.C), 256, 0, st>>>(d, descs, k); });
}
static inline int red_blocks_for(int64_t C, int sl) {
    const int ch = kRedThreads / sl;
    return (int)((C + ch - 1) / ch);
}
// reduction slices per chain: 1 (thread per chain) for few segments; 8; 32 for a handful of chains
// with hundreds of segments (cfg 5), so that the cold loads of the partial sums overlap
static inline int slices_for(const DevState &d) {
    // a full covariance of more than a handful of parameters is updated by all slices (update_cov_coop)
    const bool stage = d.p > 4 && d.p <= kCoopP;
    // one thread per chain only when there is nothing to share AND the grid would still fill the GPU:
    // the sliced layouts also give the next proposal a warp of its own (accept_kernel, task split)
    if (!stage && (d.use_ssum || d.S * d.G <= 16) && d.C >= 32768) return 1;
    return d.C <= 8 ? 32 : 8;
}
// Deferral flags of element k of an n_steps block (see run_deferred): needs the lean instantiations and
// the sliced layout on both sides; d is the handle's state (not a gradient view).  EXTMCMC_DEFER=0: off.
int step_deferral_flags(const DevState &d, int k, int n_steps) {
    static const bool on = [] { const char *e = getenv("EXTMCMC_DEFER"); return !e || atoi(e) != 0; }();
    if (!(on && d.lean && slices_for(d) >= 8)) return 0;
    return (k > 0 ? kFlagConsume : 0) | (k + 1 < n_steps ? kFlagDefer : 0);
}
void launch_accept(const DevState &d0, const StepDesc *descs, int k, int fuse_next, int flags, cudaStream_t st,
                   bool from_cache) {
    // from_cache: no sweep ran for this element; the sums of its proposal are the cached per-group sums
    // of the current state, read as a partial buffer with one segment per group.  The thread layout is
    // the one the handle's real state gives (the deferral flags were derived from it).
    DevState d = d0;
    if (from_cache) { d.partial = d0.dsum_cur; d.S = 1; d.use_ssum = 0; d.p2p = 0; flags |= kFlagNoSweep; }
    // PDL attribute: the accept kernel's prologue overlaps the tail of the sweep
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (pdl_mask() >> 1) & 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const int sl = slices_for(d0);
    cfg.gridDim = dim3(red_blocks_for(d.C, sl));
    with_spec(d, [&](auto sp) {
        using SP = decltype(sp);
        if (sl == 32) cudaLaunchKernelEx(&cfg, accept_kernel<32, SP>, d, descs, k, fuse_next, flags);
        else if (sl == 8) cudaLaunchKernelEx(&cfg, accept_kernel<8, SP>, d, descs, k, fuse_next, flags);
        else cudaLaunchKernelEx(&cfg, accept_kernel<1, SP>, d, descs, k, fuse_next, flags);
    });
}
void launch_grad_finalize(const DevState &d, const double *src, double *ll_out, double *grad_out,
                          cudaStream_t st) {
    grad_finalize_kernel<<<(int)((d.C + 127) / 128), 128, 0, st>>>(d, src, ll_out, grad_out);
}
void launch_mala_propose(const DevState &d, const StepDesc *descs, int k, int finalize_cur, double *ll_scratch,
                         int flags, cudaStream_t st) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)((d.C + kMalaChains - 1) / kMalaChains));
    cfg.blockDim = dim3(kMalaChains * kMalaSlices);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (pdl_mask() >> 1) & 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    with_spec(d, [&](auto sp) { cudaLaunchKernelEx(&cfg, mala_propose_kernel<decltype(sp)>, d, descs, k, finalize_cur, ll_scratch, flags); });
}
void launch_mala_accept(const DevState &d, const StepDesc *descs, int k, int finalize_prop, int fuse_next,
                        int flags, cudaStream_t st) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)((d.C + kMalaChains - 1) / kMalaChains));
    cfg.blockDim = dim3(kMalaChains * kMalaSlices);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (pdl_mask() >> 1) & 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    with_spec(d, [&](auto sp) { cudaLaunchKernelEx(&cfg, mala_accept_kernel<decltype(sp)>, d, descs, k, finalize_prop, fuse_next, flags); });
}
void launch_chol_factor(double *S, double *L, int n, int64_t stride, int64_t count, cudaStream_t st) {
    chol_factor_kernel<<<(int)((count + 127) / 128), 128, 0, st>>>(S, L, n, stride, count);
}
void launch_prepare_current(const DevState &d, cudaStream_t st) {
    prepare_current_kernel<<<blocks_for(d.C), 256, 0, st>>>(d);
}
void launch_reduce_group_sums(const DevState &d, double *out, cudaStream_t st) {
    const int64_t n = (int64_t)2 * d.G * d.C;
    reduce_group_sums_kernel<<<(int)((n + 255) / 256), 256, 0, st>>>(d, out);
}
void launch_reduce_partials(const DevState &d, cudaStream_t st) {
    if (d.S * d.G > 16)
        reduce_partials_kernel<8><<<red_blocks_for(d.C, 8), 256, 0, st>>>(d);
    else
        reduce_partials_kernel<1><<<red_blocks_for(d.C, 1), 256, 0, st>>>(d);
}
void launch_reduce_push(const DevState &d, const StepDesc *descs, int k, cudaStream_t st) {
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(256);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = (pdl_mask() >> 1) & 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    if (d.S * d.G > 16) {
        cfg.gridDim = dim3(red_blocks_for(d.C, 8));
        cudaLaunchKernelEx(&cfg, reduce_push_kernel<8>, d, descs, k);
    } else {
        cfg.gridDim = dim3(red_blocks_for(d.C, 1));
        cudaLaunchKernelEx(&cfg, reduce_push_kernel<1>, d, descs, k);
    }
}
void launch_finalize_loglik(const DevState &d, double *ll_out, cudaStream_t st) {
    finalize_loglik_kernel<<<blocks_for(d.C), 256, 0, st>>>(d, ll_out);
}
void launch_generate_obs_normal(double *obs, int64_t first, int64_t n, double mean, double sd,
                                uint64_t seed, int num_sms, cudaStream_t st) {
    generate_obs_normal_kernel<<<num_sms * 8, 256, 0, st>>>(obs, first, n, mean, sd, seed);
}
void launch_flush_l2(double *buf, int64_t n, int num_sms, cudaStream_t st) {
    flush_l2_kernel<<<num_sms * 8, 256, 0, st>>>(buf, n, 1.0);
}
void launch_dmma_peak(double *out, int iters, int num_sms, cudaStream_t st) {
    dmma_peak_kernel<<<num_sms * 8, 256, 0, st>>>(out, iters, 1.0000001, 1e-9);
}
void launch_fp64_peak(double *out, int iters, int num_sms, cudaStream_t st) {
    fp64_peak_kernel<<<num_sms * 8, 256, 0, st>>>(out, iters, 1.0000001, 1e-9);
}

}  // namespace extmcmc
