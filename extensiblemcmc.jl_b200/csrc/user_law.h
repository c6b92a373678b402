// Host side of the user-defined laws (EXTMCMC_LAW_USER): run-time compilation of the user's source
// with the sweep template (NVRTC, loaded with dlopen), the loaded kernels of one handle, the planner
// and the launch of sweep + finalize (user_law.cu).
#pragma once
#include <cstdint>
#include <string>
#include <cuda_runtime.h>
#include "sweep.h"
#include "sweep_user.cuh"
#include "dev_state.cuh"

namespace extmcmc {

// Widest chunk the library picks for a forward-mode law with more than kUserMaxForwardParams
// parameters: every sample law compiles without spills at it up to P = 64 (DESIGN K6).
constexpr int kUserAutoChunk = 5;

// The chunk width K of a forward-mode law of P parameters: chunk = 0 is the library's choice (P <= 16:
// K = P, the unchunked program; above, the balanced K = ceil(P / ceil(P / kUserAutoChunk))), otherwise
// a width in 1..min(kUserMaxChunk, P) that makes at most kUserMaxChunks chunks.  EXTMCMC_OK, or
// EXTMCMC_EINVAL with err.  The caller checks 1 <= P <= kUserMaxParams.
int32_t user_law_chunk(int P, int chunk, int &K, std::string &err);

// Compiles every instantiation the planner can pick for (P, D, mode) to an sm_100a cubin, or takes it
// from the process-wide cache keyed by the exact NVRTC input.  mode: a UserGrad (sweep_user.cuh; the
// caller resolves the chunk width K of kUserGradForward with user_law_chunk; other modes ignore K).
// flags: EXTMCMC_USER_* (EXTMCMC_USER_THETA_TERM compiles the law's logpdf_theta into the sweeps).
// theta_only: coordinates the rows do not read (bit k = coordinate k; needs EXTMCMC_USER_THETA_TERM):
// the sweeps then sum rows only and the parameter-only kernels add the term.
// log: NVRTC + ptxas log.  Returns EXTMCMC_OK, EXTMCMC_EINVAL (the source does not compile) or
// EXTMCMC_EUNSUPPORTED (no NVRTC).
int32_t user_law_compile(const char *source, int P, int D, int mode, int K, int flags, uint64_t theta_only,
                         std::string &log, std::string &cubin, uint64_t *input_hash);

constexpr int kUserThetaNT = 128;   // threads per CTA of the parameter-only kernels (a chain each)

struct UserLaw {
    bool loaded = false;
    bool grad = false;                      // the law has gradient kernels (mode != kUserValue)
    int mode = kUserValue;                  // UserGrad: how they compute it
    int P = 0, D = 0;
    int K = 0, n_chunks = 1;                // forward mode: chunk width and gradient sweeps (K = P: one)
    uint64_t theta_only = 0;                // coordinates the rows do not read (0: none declared)
    uint64_t hash = 0;                      // FNV-1a of the NVRTC input (checkpoint blobs record it)
    cudaLibrary_t lib = nullptr;
    // [R = 1, 2, 4][slot]: slot 0 the value kernel, slot 1 + c the gradient kernel of chunk c
    // (hand-written or forward mode)
    cudaKernel_t chains[3][1 + kUserMaxChunks] = {};
    cudaKernel_t lanes[1 + kUserMaxChunks] = {};   // [slot]
    int occ_chains[3] = {1, 1, 1}, occ_lanes = 1;   // resident CTAs per SM
    cudaKernel_t theta[2] = {};             // theta_only: the parameter-only kernels, [value, gradient]
};

// Loads the cubin into u (replacing what u held).  Returns a CUDA error.
cudaError_t user_law_load(UserLaw &u, const std::string &cubin, int P, int D, int mode, int K, uint64_t theta_only,
                          uint64_t hash);
void user_law_unload(UserLaw &u);

SweepPlan plan_sweep_user(const UserLaw &u, int64_t C, int64_t n_obs, int force_variant, int num_sms);
// Kernel launches of one sweep: the sweep kernel (one per chunk of a gradient) and the finalize
// (a law with theta_only: + the parameter-only kernel, when the sweep finishes ll)
inline int user_sweep_launches(const UserLaw &u, bool grad, bool finish = true) {
    return (grad ? u.n_chunks : 1) + 1 + (u.theta_only && finish ? 1 : 0);
}
// sweep(s) + fixed-order finalize: ll_dst[C], grad_dst[P][C] (grad only).  A law with theta_only
// finalizes the row sums into rsum ([1 + P][C]: R, then Rg with grad) and, unless ll_dst is NULL, adds
// the parameter-only term from there (launch_theta_user).
cudaError_t launch_sweep_user(const SweepPlan &pl, const UserLaw &u, const UserSweepArgs &a, bool grad,
                              double *ll_dst, double *grad_dst, double *rsum, cudaStream_t st);
// The parameter-only kernel of a law with theta_only: a.ll (and a.grad with grad) from a.rsum and a.theta
cudaError_t launch_theta_user(const UserLaw &u, const UserThetaArgs &a, bool grad, cudaStream_t st);

// ---- user-defined priors (EXTMCMC_PRIOR_USER, prior_user.cuh) -------------------------------------
constexpr int kUserPriorNT = 128;        // threads per CTA of the prior kernels (a chain each)
constexpr int kUserPriorMaxCoords = 64;  // p_u of a user prior (MALA; the random walks stop at kMaxCoords)

// Compiles the prior's kernels for (PU, mode) -- mode: a UserGrad; the random-walk kernel when
// PU <= kMaxCoords, the gradient kernel when mode != kUserValue -- through the cache of user_law_compile.
// EXTMCMC_OK, EXTMCMC_EINVAL (does not compile) or EXTMCMC_EUNSUPPORTED (no NVRTC).
int32_t user_prior_compile(const char *source, int PU, int mode, std::string &log, std::string &cubin);

struct UserPrior {
    bool loaded = false;
    int mode = kUserValue;      // UserGrad of the compiled program
    int PU = 0;
    cudaLibrary_t lib = nullptr;
    cudaKernel_t rw = nullptr;    // draw + redraw loop + lp of proposal and current state
    cudaKernel_t grad = nullptr;  // lp and gradient of a state (mode != kUserValue)
};
cudaError_t user_prior_load(UserPrior &p, const std::string &cubin, int PU, int mode);
void user_prior_unload(UserPrior &p);
// The kernels on element k of descs: the draw (writes prop_loc, n_used, prior_dev [2][C]); lp and gradient of
// the state src into prior_dev + s (1 + PU) C (s = 0 the current state, 1 the proposal)
cudaError_t launch_prior_rw(const UserPrior &p, const DevState &d, const StepDesc *descs, int k, cudaStream_t st);
cudaError_t launch_prior_grad(const UserPrior &p, const DevState &d, const StepDesc *descs, int k, const double *src,
                              int s, cudaStream_t st);

}  // namespace extmcmc
