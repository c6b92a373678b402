// Host side of the user-defined laws (EXTMCMC_LAW_USER): run-time compilation of the user's source
// with the sweep template (NVRTC, loaded with dlopen), the loaded kernels of one handle, the planner
// and the launch of sweep + finalize (user_law.cu).
#pragma once
#include <cstdint>
#include <string>
#include <cuda_runtime.h>
#include "sweep.h"
#include "sweep_user.cuh"

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
// log: NVRTC + ptxas log.  Returns EXTMCMC_OK, EXTMCMC_EINVAL (the source does not compile) or
// EXTMCMC_EUNSUPPORTED (no NVRTC).
int32_t user_law_compile(const char *source, int P, int D, int mode, int K, int flags, std::string &log,
                         std::string &cubin, uint64_t *input_hash);

struct UserLaw {
    bool loaded = false;
    bool grad = false;                      // the law has gradient kernels (mode != kUserValue)
    int mode = kUserValue;                  // UserGrad: how they compute it
    int P = 0, D = 0;
    int K = 0, n_chunks = 1;                // forward mode: chunk width and gradient sweeps (K = P: one)
    uint64_t hash = 0;                      // FNV-1a of the NVRTC input (checkpoint blobs record it)
    cudaLibrary_t lib = nullptr;
    // [R = 1, 2, 4][slot]: slot 0 the value kernel, slot 1 + c the gradient kernel of chunk c
    // (hand-written or forward mode)
    cudaKernel_t chains[3][1 + kUserMaxChunks] = {};
    cudaKernel_t lanes[1 + kUserMaxChunks] = {};   // [slot]
    int occ_chains[3] = {1, 1, 1}, occ_lanes = 1;   // resident CTAs per SM
};

// Loads the cubin into u (replacing what u held).  Returns a CUDA error.
cudaError_t user_law_load(UserLaw &u, const std::string &cubin, int P, int D, int mode, int K, uint64_t hash);
void user_law_unload(UserLaw &u);

SweepPlan plan_sweep_user(const UserLaw &u, int64_t C, int64_t n_obs, int force_variant, int num_sms);
// Kernel launches of one sweep: the sweep kernel (one per chunk of a gradient) and the finalize
inline int user_sweep_launches(const UserLaw &u, bool grad) { return (grad ? u.n_chunks : 1) + 1; }
// sweep(s) + fixed-order finalize: ll_dst[C], grad_dst[P][C] (grad only)
cudaError_t launch_sweep_user(const SweepPlan &pl, const UserLaw &u, const UserSweepArgs &a, bool grad,
                              double *ll_dst, double *grad_dst, cudaStream_t st);

}  // namespace extmcmc
