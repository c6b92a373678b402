// The random-walk draw of one chain-step (proposal!, src/updates.jl:191-196): the Philox substream of
// (chain, mcmciter, pidx), the uniform and multiplicative steps (rand(::UniformRandomWalk),
// random_walk.jl:65-73), Box-Muller and the cached Cholesky factors L_A / L_B with the mixture's lambda
// (rand(::GaussianRandomWalk[Mix]), random_walk.jl:145-151,213-227), and the whole-vector redraw while the
// prior is exactly -Inf (updates.jl:193-195).  nvcc compiles it into the step kernels with the built-in
// priors (step_device.cuh: propose_draw); NVRTC compiles the same text into the program of a user-defined
// prior (prior_user.cuh), which evaluates the user's logprior inside the redraw loop.
#pragma once
#ifndef __CUDACC_RTC__
#include <cmath>
#include <cstdint>
#endif
#include "dev_state.cuh"
#include "philox.cuh"

namespace extmcmc {

// ---- accessors ---------------------------------------------------------------------------------
struct StrideGet {            // q[i * stride] (one chain's column of an SoA array)
    const double *p;
    int64_t stride;
    __device__ __forceinline__ double operator()(int i) const { return p[(int64_t)i * stride]; }
};
struct CoordGet {             // theta[coords[i]] of one chain
    const double *col;        // theta + c
    const int32_t *coords;
    int64_t C;
    __device__ __forceinline__ double operator()(int i) const { return col[(int64_t)coords[i] * C]; }
};
// column-major n x n matrix, either shared by all chains (stride 1) or per chain (stride C, + c)
struct MatRef {
    double *p;
    int64_t stride;
    __device__ __forceinline__ double get(int idx) const { return p[(int64_t)idx * stride]; }
    __device__ __forceinline__ void set(int idx, double v) const { p[(int64_t)idx * stride] = v; }
};

__device__ __forceinline__ MatRef mat_LA(const DevUpdate &u) { return MatRef{u.LA, 1}; }
__device__ __forceinline__ MatRef mat_LB(const DevUpdate &u, int64_t C, int64_t c) { return MatRef{u.LB + c, C}; }

// Writes prop_loc and n_used of chain c.  kern: the update's transition kernel; log_prior(get): the
// prior of the local proposal read through a StrideGet (the redraw loop ends when it is not -Inf).
template <class LogPrior>
__device__ __forceinline__ void rw_draw(const DevState &d, const StepDesc &sd, const DevUpdate &u, int64_t c, int kern,
                                        LogPrior log_prior) {
    const int n = u.n_coords;
    const int64_t C = d.C;
    const CoordGet th{d.theta + c, u.coords, C};
    const StrideGet prop{d.prop_loc + c, C};
    double *pl = d.prop_loc + c;

    uint32_t used = 0;
    if (d.rng_mode == EXTMCMC_RNG_REPLAY) {
        for (int i = 0; i < n; ++i) pl[(int64_t)i * C] = d.rp_prop[((int64_t)sd.replay_row * d.p_u_max + i) * d.gC + d.g0 + c];
    } else {
        ChainStepStream rng(d.seed, (uint64_t)(d.chain_offset + c), sd.mcmciter, sd.pidx);
        for (;;) {
            if (kern == EXTMCMC_KERNEL_RW_UNIFORM) {
                for (int i = 0; i < n; ++i) {
                    const double r = rng.next();
                    const double e = u.eps[(int64_t)i * C + c];
                    const double a = -e, b = e;
                    const double U = a + (b - a) * r;  // rand(Uniform(-eps, eps))
                    const double t = th(i);
                    pl[(int64_t)i * C] = u.pos[i] ? t * exp(U) : t + U;  // random_walk.jl:72
                }
            } else {
                // rand(rw::GaussianRandomWalk[Mix]) random_walk.jl:145-151,213-227
                bool useB = false;
                if (kern == EXTMCMC_KERNEL_RW_GAUSS_MIX) useB = rng.next() <= sd.lambda;  // Bernoulli(lambda)
                double *z = d.gw + c;
                for (int q = 0; q < n; q += 2) {  // randn via Box-Muller on the uniform stream
                    const double u1 = rng.next(), u2 = rng.next();
                    const double rad = sqrt(-2.0 * log(u1));
                    double sn, cs;
                    sincospi(2.0 * u2, &sn, &cs);
                    z[(int64_t)q * C] = rad * cs;
                    if (q + 1 < n) z[(int64_t)(q + 1) * C] = rad * sn;
                }
                const MatRef L = useB ? mat_LB(u, C, c) : mat_LA(u);
                if (isnan(L.get(0))) {
                    *d.err_flag = 1;  // reference: PosDefException from MvNormal(theta, Sigma)
                    for (int i = 0; i < n; ++i) pl[(int64_t)i * C] = NAN;
                    break;
                }
                for (int i = 0; i < n; ++i) {
                    const double x = th(i);
                    double t = u.pos[i] ? log(x) : x;
                    double a = 0.0;
                    for (int k = 0; k <= i; ++k) a += L.get(i + k * n) * z[(int64_t)k * C];
                    t = a + t;
                    pl[(int64_t)i * C] = u.pos[i] ? exp(t) : t;
                }
            }
            // whole-vector redraw while the prior is exactly -Inf (updates.jl:193-195)
            if (!(log_prior(prop) == -INFINITY)) break;
            if (rng.j > 60000u) break;
        }
        used = rng.j;
    }
    d.n_used[c] = used;
}

}  // namespace extmcmc
