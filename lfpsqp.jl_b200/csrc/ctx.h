// ctx.h -- the library context behind the opaque lfpsqp_ctx handle.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <string>
#include <vector>
#include "../../include/lfpsqp_b200.h"

struct LargeState;  // large-n mode workspace (large.cu)

struct CommState {           // communicator of a column-sharded solve (comm.cu); world <= 1 means single GPU
  void *nccl = nullptr;      // ncclComm_t (large messages: the m x m Gram)
  int rank = 0, world = 0;
  // peer-memory all-reduce for the small latency-bound messages (m-vectors, packed scalars): every rank exports one
  // buffer over CUDA IPC; kernels store/load through the NVLink-mapped peer pointers
  double *peer_local = nullptr;          // this rank's region (cudaMalloc)
  double *peer_map[8] = {nullptr};       // peer_map[r] = rank r's region mapped into this process (peer_map[rank] = peer_local)
  bool peer_ready = false;
  unsigned long long epoch = 0;
};

struct lfpsqp_ctx {
  int device = 0, sm_count = 148, smem_optin = 232448;
  cudaStream_t own_stream = nullptr, stream = nullptr, pipe[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  unsigned long long *work_counter = nullptr;
  double last_ms = 0.0;
  int64_t last_launches = 0;
  int last_kernel[4] = {-1, 0, 0, 0};   // lfpsqp_last_kernel: {kind, LW, NPL, SPARSE} of the last batched launch
  std::string err;
  std::vector<void *> bufs;  // grow-only device arena, one slot per role (no allocation inside solve loops)
  std::vector<size_t> caps;
  LargeState *large = nullptr;
  CommState comm;
  // multi-GPU context (lfpsqp_ctx_create_multi): one child ctx per device; batched solves shard contiguous instance ranges
  // over the children from one host call (one host thread per device, no collective).  Empty for a single-GPU ctx.
  std::vector<lfpsqp_ctx *> children;
  // caller-supplied noise of the next device-family solve (lfpsqp_ctx_set_noise): host pointer owned by the caller
  const double *noise_host = nullptr; int64_t noise_T = 0, noise_N = 0, noise_B = 0;
  std::vector<double> bnd_host;   // host copy of the bound table of the current batched call: [kind | q | r | s | t] x NA

  int fail(int code, const char *fmt, ...);
  int cuda_fail(cudaError_t e, const char *what);
  void *arena(int slot, size_t bytes);
};

void lfpsqp_large_release(lfpsqp_ctx *c);
