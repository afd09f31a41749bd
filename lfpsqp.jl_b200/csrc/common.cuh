// common.cuh -- shared device helpers for the LFPSQP B200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include "../../include/lfpsqp_b200.h"

#define LFPSQP_DEV __device__ __forceinline__

namespace lfpsqp {

// NaN-propagating max, as Julia's norm(x, Inf)
LFPSQP_DEV double pmax(double a, double b) { return (a > b || isnan(a)) ? a : b; }

// One warp cooperating on one instance.  Reductions are xor-butterflies so that every lane holds the
// bitwise-identical result (control flow stays warp-uniform without a broadcast).
struct WarpGroup {
  static constexpr int SIZE = 32;
  int lane;
  LFPSQP_DEV explicit WarpGroup(int l) : lane(l) {}
  LFPSQP_DEV void sync() const { __syncwarp(); }
  LFPSQP_DEV double sum(double v) const {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
  }
  LFPSQP_DEV double maxabs(double v) const {  // v already |.|
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = pmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
  }
  LFPSQP_DEV void sum2(double &a, double &b) const {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
  }
  LFPSQP_DEV int64_t bcast(int64_t v, int src) const { return __shfl_sync(0xffffffffu, v, src); }
};

// problem description handed to the family callbacks
struct FamCtx {
  int n, m, p;            // user sizes: variables, equalities c, inequalities d
  const double *prm;      // this instance's parameter blob (global memory)
  int64_t k;              // this instance's index in the launch (FamQCQP: array base + k * stride)
  lfpsqp_qcqp qp;         // FamQCQP: device pointers + batch strides (the other families ignore it)
};

struct BatchedArgs {
  int family;
  int n, m, p;            // user problem sizes
  int ineq;               // bound embedding active (optimize.jl:151-170); always 1 when p>0
  int64_t B;
  const double *fam_params; int64_t fam_stride;
  const double *x0;
  const double *bnd;      // device: [kind(as double) | q | r | s | t] x NA  (inequality_helper.jl:39-85), or null
  lfpsqp_params prm;
  double *x_out; double *obj_hist; int64_t H; int64_t *obj_len; double *lambda; lfpsqp_term *term; lfpsqp_stats *stats;
  unsigned long long *work_counter;  // persistent-CTA work queue
  // stochastic perturbation of optimize.jl:264-273 with a caller-supplied noise sequence (lfpsqp_ctx_set_noise): instance k,
  // outer iteration i < noise_T uses the N working entries at noise + (k * noise_T + i) * N ; nullptr when beta == 0
  const double *noise; int64_t noise_T;
  lfpsqp_qcqp qcqp;       // LFPSQP_FAM_QCQP: device pointers rebased to this launch's first instance, batch strides
};

// coefficient of the noise term at outer iteration i (optimize.jl:267-271); 0 beyond the supplied rows
LFPSQP_DEV double noise_coef(const lfpsqp_params &prm, int64_t i, int64_t T) {
  if (!(prm.beta > 0.0) || i >= T) return 0.0;
  return prm.t_beta > 0 ? prm.beta * fmax(1.0 - (double)i / (double)prm.t_beta, 0.0) : prm.beta;
}

}  // namespace lfpsqp
