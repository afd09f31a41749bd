// batched_reg.cu -- instantiations + launcher of the register-resident batched solver (batched_reg.cuh).
#include <stdlib.h>
#include <string.h>
#include "ctx.h"
#include "batched_reg.cuh"
#include "launch.cuh"

using namespace lfpsqp;

namespace {
template <class Fam, int LW, int NPL, int ME, bool INEQ, bool SPARSE, int HEAD = 0, int MINB = 3>
int launch(lfpsqp_ctx *c, BatchedArgs &A) {
  using RS = RegSolver<Fam, LW, NPL, ME, INEQ, SPARSE, HEAD>;
  auto kern = batched_reg_kernel<Fam, LW, NPL, ME, INEQ, SPARSE, HEAD, MINB>;
  constexpr int GROUPS = REG_NT / LW;   // instances in flight per CTA
  const size_t smem = (size_t)((INEQ ? 5 * RS::NAP : 0) + GROUPS * RS::STASH_DOUBLES) * 8;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return c->cuda_fail(e, "cudaFuncSetAttribute (batched_reg_kernel)");
  int resident = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, REG_NT, smem);
  if (e != cudaSuccess || resident < 1) return c->cuda_fail(e, "occupancy query (batched_reg_kernel)");
  const int64_t grid = persistent_grid(c, A, resident, GROUPS);
  return launch_batched_kernel(c, kern, grid, REG_NT, smem, {2, LW, NPL, SPARSE ? 1 : 0}, "batched_reg_kernel launch", A);
}

// SPARSE layout: with element j in lane j % LW, does every lane hold at most one pair that is not a line (kind != 0)?
bool sparse_ok(const lfpsqp_ctx *c, int NA, int LW) {
  if ((int)c->bnd_host.size() < NA) return false;
  int cnt[32] = {0};
  for (int j = 0; j < NA; j++) if (c->bnd_host[j] != 0.0 && ++cnt[j % LW] > 1) return false;
  return true;
}

// line head: do slots 0 .. HEAD-1 (elements j < HEAD LW) hold only line pairs (kind 0; padding past N_A is zero)?
bool line_head_ok(const lfpsqp_ctx *c, int NA, int HEAD, int LW) {
  if ((int)c->bnd_host.size() < NA) return false;
  for (int j = 0; j < NA && j < HEAD * LW; j++) if (c->bnd_host[j] != 0.0) return false;
  return true;
}
}  // namespace

// returns LFPSQP_OK when launched, 1 when this problem shape has no register-resident instantiation (caller falls
// back to the shared-memory warp kernel), < 0 on errors.  LFPSQP_BATCHED_KERNEL=smem forces the fallback (A/B tests).
int launch_batched_reg(lfpsqp_ctx *c, BatchedArgs &A) {
  const char *force = getenv("LFPSQP_BATCHED_KERNEL");
  if (force && strcmp(force, "smem") == 0) return 1;
  if (A.prm.linesearch != 0 && !A.prm.disable_linesearch) return 1;   // exact_linesearch! lives in the shared-memory solver
  const int NA = A.n + A.p, ME = A.m + A.p;
  switch (A.family) {
    case LFPSQP_FAM_README_INEQ:
      if (ME != 1 || !A.ineq) return 1;
      if (NA <= 32) return launch<SepReadmeIneq, 16, 2, 1, true, false>(c, A);
      if (NA <= 64) {
        if (NA <= 56 && sparse_ok(c, NA, 8)) {
          if (line_head_ok(c, NA, 6, 8)) return launch<SepReadmeIneq, 8, 7, 1, true, true, 6, 2>(c, A);
          return launch<SepReadmeIneq, 8, 7, 1, true, true, 0, 2>(c, A);
        }
        return launch<SepReadmeIneq, 16, 4, 1, true, false>(c, A);
      }
      if (NA <= 128) return launch<SepReadmeIneq, 32, 4, 1, true, false>(c, A);
      return 1;
    case LFPSQP_FAM_README_EQ:
      if (ME != 1 || NA > 64) return 1;
      return A.ineq ? launch<SepReadmeEq, 16, 4, 1, true, false>(c, A) : launch<SepReadmeEq, 16, 4, 1, false, false>(c, A);
    case LFPSQP_FAM_BOXQUAD:
      if (!A.ineq || NA > 32) return 1;
      return ME == 0 ? launch<SepBoxQuad, 16, 2, 0, true, false>(c, A) : launch<SepBoxQuad, 16, 2, 1, true, false>(c, A);
    default: return 1;
  }
}
