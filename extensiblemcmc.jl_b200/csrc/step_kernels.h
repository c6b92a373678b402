// Host-side launchers of the per-chain step kernels (step_kernels.cu).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "dev_state.cuh"

namespace extmcmc {
void launch_propose(const DevState &d, const StepDesc *descs, int k, cudaStream_t st);
int step_deferral_flags(const DevState &d, int k, int n_steps);   // see run_deferred in step_kernels.cu
void launch_accept(const DevState &d, const StepDesc *descs, int k, int fuse_next, int flags, cudaStream_t st,
                   bool from_cache = false);
void launch_prepare_current(const DevState &d, cudaStream_t st);
// lower Cholesky factors of `count` column-major n x n matrices (element stride `stride`, matrix c at + c)
void launch_chol_factor(double *S, double *L, int n, int64_t stride, int64_t count, cudaStream_t st);
// user-law row-sum cache: R of an accepted random-walk proposal -> the current state's (api.cu)
void launch_rsum_commit(const DevState &d, const StepDesc *descs, int k, cudaStream_t st);
void launch_grad_finalize(const DevState &d, const double *src, double *ll_out, double *grad_out, cudaStream_t st);
void launch_mala_propose(const DevState &d, const StepDesc *descs, int k, int finalize_cur, double *ll_scratch,
                         int flags, cudaStream_t st);
void launch_mala_accept(const DevState &d, const StepDesc *descs, int k, int finalize_prop, int fuse_next,
                        int flags, cudaStream_t st);
void launch_reduce_partials(const DevState &d, cudaStream_t st);
void launch_reduce_group_sums(const DevState &d, double *out, cudaStream_t st);
void launch_reduce_push(const DevState &d, const StepDesc *descs, int k, cudaStream_t st);
void launch_finalize_loglik(const DevState &d, double *ll_out, cudaStream_t st);
void launch_generate_obs_normal(double *obs, int64_t first, int64_t n, double mean, double sd,
                                uint64_t seed, int num_sms, cudaStream_t st);
void launch_flush_l2(double *buf, int64_t n, int num_sms, cudaStream_t st);
void launch_fp64_peak(double *out, int iters, int num_sms, cudaStream_t st);
void launch_dmma_peak(double *out, int iters, int num_sms, cudaStream_t st);
}  // namespace extmcmc
