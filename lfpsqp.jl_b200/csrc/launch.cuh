// launch.cuh -- the launch steps the batched kernels share (abi.cu: tiny and warp solvers; batched_reg.cu: register solver).
#pragma once
#include <string.h>
#include <algorithm>
#include "ctx.h"
#include "common.cuh"

namespace lfpsqp {

// Grid of a persistent kernel: every resident CTA slot of the GPU, but no more CTAs than the batch needs at per_cta
// instances in flight per CTA.  The CTAs pull instance indices from the context's work counter, which starts at 0.
inline int64_t persistent_grid(lfpsqp_ctx *c, BatchedArgs &A, int resident, int per_cta) {
  cudaMemsetAsync(c->work_counter, 0, 8, c->stream);
  A.work_counter = c->work_counter;
  return std::max<int64_t>(1, std::min<int64_t>((int64_t)c->sm_count * resident, (A.B + per_cta - 1) / per_cta));
}

// kern<<<grid, threads, smem>>>(args...) on the context's stream between ev0 and ev1 (lfpsqp_last_kernel_ms), recorded
// as the call's one launch; id = {kind, LW, NPL, SPARSE} is what lfpsqp_last_kernel reports.
template <class... P, class... Args>
int launch_batched_kernel(lfpsqp_ctx *c, void (*kern)(P...), int64_t grid, int threads, size_t smem, const int (&id)[4],
                          const char *what, Args... args) {
  cudaEventRecord(c->ev0, c->stream);
  kern<<<(unsigned)grid, threads, smem, c->stream>>>(args...);
  cudaEventRecord(c->ev1, c->stream);
  c->last_launches = 1;
  memcpy(c->last_kernel, id, sizeof(c->last_kernel));
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return c->cuda_fail(e, what);
  return LFPSQP_OK;
}

}  // namespace lfpsqp
