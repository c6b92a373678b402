// Kernels of a user-defined prior (EXTMCMC_PRIOR_USER), instantiated by NVRTC around the user's
// `logprior` (+ `logprior_grad`, or a `logprior<real>` template differentiated through dual.cuh) over
// the update's EXTMCMC_PU coordinates, see user_law.cu and INTEGRATION.md.  One thread per chain.
//
// user_prior_rw: the random-walk draw of the element (rw_draw.cuh, the code the built-in priors run in
// the step kernels), with logprior inside the redraw loop; writes prop_loc and n_used and, into the
// update's prior_dev ([2][C]), logprior of the proposal and of the current state.  The nvcc propose
// kernel then assembles the full proposal and the law constants; the accept kernel reads the two terms.
//
// user_prior_grad: logprior and its gradient of a state (the current one before a MALA proposal, the
// proposal before its decision) into prior_dev + s (1 + PU) C, rows [1 + PU][C]: the value, then d/dth_i.
// EXTMCMC_PRIOR_GRAD (the program's with_grad) selects the user's logprior_grad or forward mode.
#pragma once
#include "rw_draw.cuh"
#include "dual.cuh"

namespace extmcmc {

// logprior of the update's coordinates of a state, th[i] = get(i) copied to this thread's row of `th`
template <class Get>
__device__ __forceinline__ double user_logprior(Get get, const double *pp, double *th) {
#pragma unroll
    for (int i = 0; i < EXTMCMC_PU; ++i) th[i] = get(i);
    return logprior(th, pp);
}

#if EXTMCMC_PU <= 32
__device__ __forceinline__ void user_prior_rw(const DevState &d, const StepDesc *descs, int k) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    const StepDesc sd = descs[k];
    const DevUpdate &u = d.upd[sd.pidx];
    const int64_t C = d.C;
    // the argument of logprior in shared memory: the draw's state stays in registers, nothing in local memory.
    // A thread's row is an odd number of doubles, so that the lanes of a warp reading th[i] hit distinct banks.
    constexpr int kRow = EXTMCMC_PU | 1;
    __shared__ double sh_th[EXTMCMC_PRIOR_NT * kRow];   // EXTMCMC_PRIOR_NT: threads per CTA
    double *th = sh_th + threadIdx.x * kRow;
    double lp_prop = 0.0;
    bool have = false;
    rw_draw(d, sd, u, c, u.kernel, [&](const StrideGet &prop) {
        lp_prop = user_logprior(prop, u.prior_params, th);
        have = true;
        return lp_prop;
    });
    if (!have) lp_prop = user_logprior(StrideGet{d.prop_loc + c, C}, u.prior_params, th);   // replayed proposal
    double *out = const_cast<double *>(u.prior_dev);
    out[c] = lp_prop;
    out[C + c] = user_logprior(CoordGet{d.theta + c, u.coords, C}, u.prior_params, th);
}
#endif

#if EXTMCMC_PRIOR_GRAD
__device__ __forceinline__ void user_prior_grad(const DevState &d, const StepDesc *descs, int k, const double *src, int s) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= d.C) return;
    const DevUpdate &u = d.upd[descs[k].pidx];
    const int64_t C = d.C;
    double *out = const_cast<double *>(u.prior_dev) + (int64_t)s * (1 + EXTMCMC_PU) * C + c;
    double th[EXTMCMC_PU];
#pragma unroll
    for (int i = 0; i < EXTMCMC_PU; ++i) th[i] = src[(int64_t)u.coords_dev[i] * C + c];
#if EXTMCMC_PRIOR_GRAD == 2   // EXTMCMC_USER_GRAD_FORWARD
    Dual<EXTMCMC_PU> x[EXTMCMC_PU];
#pragma unroll
    for (int i = 0; i < EXTMCMC_PU; ++i) {
        x[i] = Dual<EXTMCMC_PU>(th[i]);
        x[i].t[i] = 1.0;
    }
    const Dual<EXTMCMC_PU> r = logprior(x, u.prior_params);
    out[0] = r.v;
#pragma unroll
    for (int i = 0; i < EXTMCMC_PU; ++i) out[(int64_t)(1 + i) * C] = r.t[i];
#else
    double g[EXTMCMC_PU];
#pragma unroll
    for (int i = 0; i < EXTMCMC_PU; ++i) g[i] = 0.0;
    out[0] = logprior_grad(th, u.prior_params, g);
#pragma unroll
    for (int i = 0; i < EXTMCMC_PU; ++i) out[(int64_t)(1 + i) * C] = g[i];
#endif
}
#endif

}  // namespace extmcmc
