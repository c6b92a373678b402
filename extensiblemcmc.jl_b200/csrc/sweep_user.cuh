// Likelihood sweep of a user-defined law (EXTMCMC_LAW_USER): the kernel template that NVRTC
// instantiates at run time around the user's `Law`, `set_parameters` and `logpdf` (+ `logpdf_grad`,
// or forward-mode derivatives of a `Law<real>` template through dual.cuh), see user_law.cu and
// INTEGRATION.md.  nvcc compiles this header too (user_law.cu: the argument
// struct and the shape constants the host planner shares with the kernel); the template is only
// instantiated in the NVRTC program, where the user's functions are visible.
//
// grid = (observation segments S, chain groups).  A CTA streams the rows of its segment HBM/L2 ->
// shared memory with 1-D TMA bulk copies (tma.cuh) in a ring of kUserStages tiles.  A thread holds
// R chains: for each it calls set_parameters once on the evaluated state theta[P][C] and keeps the
// Law in registers for the whole sweep, then walks the rows j = lane (mod L) of every tile:
//   L = 1  ("chains"): every thread of the CTA reads the same row (broadcast), R chains per thread;
//   L = 32 ("lanes") : a warp shares one chain, lane l takes rows l, l + 32, ... of each tile.
// Each thread accumulates its rows in order; the lanes of a chain are combined by a fixed xor-shuffle
// tree; per-segment sums go to ll_part[S][C] and g_part[S][P][C], which the finalize kernel
// (user_law.cu) adds in segment order.  No atomics: the result does not depend on the schedule.
//
// G selects what a row contributes: kUserValue calls logpdf; kUserGradHand calls the user's
// logpdf_grad; kUserGradForward runs LawT = Law<Dual<K>>: theta enters set_parameters as duals seeded
// with the unit vectors of coordinates [CI*K, CI*K + K), so logpdf returns the row's value and those K
// partial derivatives, which go to the same accumulators as the hand-written gradient's.  K = P is one
// sweep for the whole gradient; K < P is chunk CI of ceil(P/K) sweeps (ForwardDiff's chunk mode).  A
// tangent component is the same expression whatever K is, so the chunks together produce the bits of
// the unchunked sweep.  The chunk is a template parameter on purpose: with a compile-time seed the
// tangents of every field copied from theta fold into immediates.
#pragma once
#ifndef __CUDACC_RTC__
#include <cstdint>
#endif
#include "dual.cuh"
#include "tma.cuh"

namespace extmcmc {

constexpr int kUserNT = 128;             // threads per CTA, both mappings
constexpr int kUserStages = 3;           // tiles in flight per CTA
constexpr int kUserTileDoubles = 1024;   // shared memory per stage: 8 KB
constexpr int kUserMaxParams = 64;       // n_params of a user law (register file: theta, Law, gradient)
constexpr int kUserMaxObsDim = 64;       // obs_dim of a user law (>= 16 rows per tile)

// Rows per tile: an even number, so that a tile is a whole number of 16-byte units whatever D is
// (the device buffer holds an even number of rows, zero-padded).
__host__ __device__ constexpr int user_tile_rows(int D) { return (kUserTileDoubles / D) & ~1; }

constexpr int kUserMaxForwardParams = 16;   // n_params of an unchunked forward-mode law (P + 1 doubles per field)
constexpr int kUserMaxChunk = 16;           // tangents per chunk of a chunked forward-mode law
constexpr int kUserMaxChunks = 16;          // chunk sweeps per gradient (bounds the JIT)

// What a sweep computes, and how a law provides its gradient (the values of with_grad, extmcmc.h)
enum UserGrad : int { kUserValue = 0, kUserGradHand = 1, kUserGradForward = 2 };

// Doubles a thread holds per chain, for the register budget: a Law of ~P doubles and ll, plus the P
// gradient accumulators with a gradient; under forward mode with chunk width K every field of the
// Law<Dual<K>> holds K + 1 doubles: P such fields and the accumulators make (P + 1)(K + 1).
__host__ __device__ constexpr int user_chain_doubles(int P, int grad, int K) {
    return grad == kUserGradForward ? (P + 1) * (K + 1) : grad ? 2 * P + 1 : P + 1;
}
// Chains per thread the "chains" mapping may use: the accumulators (ll, and the gradient with GRAD)
// of all R chains live in registers next to the R Laws.  grad: a UserGrad, K: the chunk width of forward
// mode (the kernels of a law are planned for the mode it was compiled in: its value kernels run at the
// R of its gradient kernels).
__host__ __device__ constexpr int user_max_R(int P, int grad, int K) {
    return user_chain_doubles(P, grad, K) * 4 <= 40 ? 4 : user_chain_doubles(P, grad, K) * 2 <= 40 ? 2 : 1;
}

struct UserSweepArgs {
    const double *obs;     // [n_pad][D] row-major, n_pad = n_obs rounded up to even (zero rows)
    int64_t n_obs;
    const double *theta;   // [P][C] the evaluated state (proposal or current)
    int64_t C;
    double *ll_part;       // [S][C]
    double *g_part;        // [S][P][C] (GRAD)
    int32_t *err_flag;     // set when a chain's set_parameters returns false
    int S;
};

#ifdef __CUDACC_RTC__
#ifdef EXTMCMC_THETA_TERM
// Adds the law's parameter-only term (EXTMCMC_USER_THETA_TERM) to a chain's sums: its value to ll and,
// with a gradient, its derivatives in the coordinates of the sweep's accumulators to g[0..NG-1] --
// logpdf_theta_grad on a zeroed t (hand-written), or the tangents of logpdf_theta on the Law<Dual<K>> of
// the chunk (forward mode).  Each sum gets one addition: ll = fl(rows + term), g[k] = fl(rows_k + t_k).
template <int G, int NG, class LawT>
__device__ __forceinline__ void user_add_theta_term(const LawT &L, double &ll, double *g) {
    if constexpr (G == kUserGradForward) {
        const auto t = logpdf_theta(L);
        ll += t.v;
#pragma unroll
        for (int k = 0; k < NG; ++k) g[k] += t.t[k];
    } else if constexpr (G == kUserGradHand) {
        double t[NG];
#pragma unroll
        for (int k = 0; k < NG; ++k) t[k] = 0.0;
        ll += logpdf_theta_grad(L, t);
#pragma unroll
        for (int k = 0; k < NG; ++k) g[k] += t[k];
    } else {
        ll += logpdf_theta(L);
    }
}
#endif

// K, CI: chunk width and chunk index of a forward-mode sweep (LawT = Law<Dual<K>>); chunk 0 writes
// ll_part and raises err_flag, every chunk writes only its own rows g_part[S][CI*K ..][C].
// With EXTMCMC_THETA_TERM the CTAs of segment 0 add the law's parameter-only term to the sums of their
// own rows (user_add_theta_term).
template <class LawT, int P, int D, int R, int L, int G, int K = P, int CI = 0>
__device__ __forceinline__ void user_sweep(const UserSweepArgs &a) {
    constexpr bool GRAD = G != kUserValue;
    constexpr bool FWD = G == kUserGradForward;
    constexpr int NG = FWD ? K : P;          // gradient accumulators per chain
    constexpr int K0 = FWD ? CI * K : 0;     // first coordinate they belong to
    constexpr bool WRITE_LL = K0 == 0;
    static_assert(K0 < P && K <= P, "chunk out of range");
    constexpr int TR = user_tile_rows(D), ST = kUserStages;
    constexpr int CPB = kUserNT / L * R;   // chains per CTA
    static_assert(L == 1 || R == 1, "the lanes mapping holds one chain per warp");
    __shared__ __align__(128) double tile[ST][TR * D];
    __shared__ __align__(8) uint64_t bar[ST];
    const int tid = threadIdx.x;
    const int lane = L == 1 ? 0 : (tid & (L - 1));
    const int seg = blockIdx.x;
    const int64_t C = a.C;
    const int64_t cbase = (int64_t)blockIdx.y * CPB;

    // segment bounds on even rows: every bulk copy starts 16-byte aligned
    const int64_t n_pairs = (a.n_obs + 1) >> 1;
    const int64_t lo = 2 * ((int64_t)seg * n_pairs / a.S);
    int64_t hi = 2 * ((int64_t)(seg + 1) * n_pairs / a.S);
    if (hi > a.n_obs) hi = a.n_obs;
    const int64_t len = hi - lo;
    const int n_tiles = (int)((len + TR - 1) / TR);

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < ST; ++s) mbar_init(&bar[s], 1);
        mbar_fence_init();
    }
    __syncthreads();
    auto issue = [&](int t) {
        const int st = t % ST;
        const int64_t off = (int64_t)t * TR;
        const int cnt = (int)((len - off) < (int64_t)TR ? (len - off) : (int64_t)TR);
        const uint32_t bytes = (uint32_t)((cnt + 1) >> 1) * (16u * D);   // pairs of rows
        mbar_expect_tx(&bar[st], bytes);
        bulk_g2s(&tile[st][0], a.obs + (lo + off) * D, bytes, &bar[st]);
    };
    if (tid == 0)
        for (int t = 0; t < ST && t < n_tiles; ++t) issue(t);

    // Only the (constant) observations were touched so far.  The evaluated state is written by the
    // preceding step kernel: wait for it, then let our own successor's prologue start.
    griddep_wait();
    griddep_launch_dependents();

    LawT law[R];
    bool ok[R];
    double acc[R];
    double g[GRAD ? R : 1][GRAD ? NG : 1];
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int64_t c = cbase + (L == 1 ? (int64_t)r * kUserNT + tid : (int64_t)(tid / L));
        if constexpr (FWD) {
            Dual<K> th[P];
#pragma unroll
            for (int k = 0; k < P; ++k) {
                th[k].v = c < C ? a.theta[(int64_t)k * C + c] : 0.0;
#pragma unroll
                for (int j = 0; j < K; ++j) th[k].t[j] = K0 + j == k ? 1.0 : 0.0;
            }
            ok[r] = c < C && set_parameters(law[r], th);
        } else {
            double th[P];
#pragma unroll
            for (int k = 0; k < P; ++k) th[k] = c < C ? a.theta[(int64_t)k * C + c] : 0.0;
            ok[r] = c < C && set_parameters(law[r], th);
        }
        acc[r] = 0.0;
        if (GRAD) {
#pragma unroll
            for (int k = 0; k < NG; ++k) g[r][k] = 0.0;
        }
    }

    for (int t = 0; t < n_tiles; ++t) {
        const int st = t % ST;
        mbar_wait(&bar[st], (uint32_t)(t / ST) & 1u);
        const int64_t off = (int64_t)t * TR;
        // rows beyond the segment (and the zero padding) never reach logpdf
        const int cnt = (int)((len - off) < (int64_t)TR ? (len - off) : (int64_t)TR);
        const double *xs = &tile[st][0];
#pragma unroll 4
        for (int j = lane; j < cnt; j += L) {
            const double *x = xs + j * D;
#pragma unroll
            for (int r = 0; r < R; ++r) {
                if (!ok[r]) continue;
                if constexpr (FWD) {
                    const auto v = logpdf(law[r], x);
                    acc[r] += v.v;
#pragma unroll
                    for (int k = 0; k < NG; ++k) g[r][k] += v.t[k];
                } else if constexpr (GRAD) {
                    acc[r] += logpdf_grad(law[r], x, g[r]);
                } else {
                    acc[r] += logpdf(law[r], x);
                }
            }
        }
        __syncthreads();   // everyone is done with this stage before it is refilled
        if (tid == 0 && t + ST < n_tiles) issue(t + ST);
    }

    const double nan = __longlong_as_double(0x7ff8000000000000ll);
#pragma unroll
    for (int r = 0; r < R; ++r) {
        const int64_t c = cbase + (L == 1 ? (int64_t)r * kUserNT + tid : (int64_t)(tid / L));
#ifdef EXTMCMC_THETA_TERM
        // Segment 0 adds the term once per chain to the sums of its rows.  The lanes of a chain are reduced
        // first: all of them then hold the sums, and all evaluate the term (the warp stays converged), and
        // the term is not held in registers across the shuffles.
        constexpr int LR = 1;   // the lanes are reduced here
        if (L > 1) {
#pragma unroll
            for (int o = L / 2; o > 0 && WRITE_LL; o >>= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
#pragma unroll
            for (int k = 0; k < NG && GRAD; ++k) {
                if (K0 + k >= P) break;
#pragma unroll
                for (int o = L / 2; o > 0; o >>= 1) g[r][k] += __shfl_xor_sync(0xffffffffu, g[r][k], o);
            }
        }
        if (seg == 0 && c < C && ok[r]) user_add_theta_term<G, NG>(law[r], acc[r], g[r]);
#else
        constexpr int LR = L;
#endif
        if constexpr (WRITE_LL) {
            double v = acc[r];
            if (LR > 1) {
#pragma unroll
                for (int o = L / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            }
            if (lane == 0 && c < C) a.ll_part[(int64_t)seg * C + c] = ok[r] ? v : nan;
        }
        if (GRAD) {
#pragma unroll
            for (int k = 0; k < NG; ++k) {
                if (K0 + k >= P) break;   // the tangents past P of a narrower last chunk: seeded zero, not written
                double w = g[r][k];
                if (LR > 1) {
#pragma unroll
                    for (int o = L / 2; o > 0; o >>= 1) w += __shfl_xor_sync(0xffffffffu, w, o);
                }
                if (lane == 0 && c < C) a.g_part[((int64_t)seg * P + K0 + k) * C + c] = ok[r] ? w : nan;
            }
        }
        if (WRITE_LL && lane == 0 && c < C && !ok[r] && seg == 0) *a.err_flag = 1;
    }
}
#endif

}  // namespace extmcmc
