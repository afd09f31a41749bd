// batched_reg.cu -- instantiations + launcher of the register-resident batched solver (batched_reg.cuh).
#include <stdlib.h>
#include <string.h>
#include "ctx.h"
#include "batched_reg.cuh"

using namespace lfpsqp;

namespace {
template <class Fam, int LW, int NPL, int ME, bool INEQ, bool SPARSE, int NT = 128, int MINB = 3>
int launch(lfpsqp_ctx *c, BatchedArgs &A) {
  using RS = RegSolver<Fam, LW, NPL, ME, INEQ, SPARSE>;
  auto kern = batched_reg_kernel<Fam, LW, NPL, ME, INEQ, SPARSE, NT, MINB>;
  constexpr int GROUPS = NT / LW;   // instances in flight per CTA
  const size_t smem = (size_t)((INEQ ? 5 * RS::NAP : 0) + GROUPS * RS::STASH_DOUBLES) * 8;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return c->cuda_fail(e, "cudaFuncSetAttribute (batched_reg_kernel)");
  int resident = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, NT, smem);
  if (e != cudaSuccess || resident < 1) return c->cuda_fail(e, "occupancy query (batched_reg_kernel)");
  c->round_instances = (int64_t)c->sm_count * resident * GROUPS;
  if (c->query_round) return LFPSQP_OK;
  int64_t grid = (int64_t)c->sm_count * resident, need = (A.B + GROUPS - 1) / GROUPS;
  if (grid > need) grid = need;
  if (grid < 1) grid = 1;
  cudaMemsetAsync(c->work_counter, 0, 8, c->stream);
  A.work_counter = c->work_counter;
  cudaEventRecord(c->ev0, c->stream);
  kern<<<(unsigned)grid, NT, smem, c->stream>>>(A);
  cudaEventRecord(c->ev1, c->stream);
  c->last_launches = 1;
  c->last_cfg_warps = NT / 32; c->last_cfg_grid = (int)grid; c->last_cfg_smem = (int)smem; c->last_cfg_resident = resident;
  c->last_kernel[0] = 2; c->last_kernel[1] = LW; c->last_kernel[2] = NPL; c->last_kernel[3] = SPARSE ? 1 : 0;
  e = cudaGetLastError();
  if (e != cudaSuccess) return c->cuda_fail(e, "batched_reg_kernel launch");
  return LFPSQP_OK;
}

// SPARSE layout: with element j in lane j % LW, does every lane hold at most one pair that is not a line (kind != 0)?
bool sparse_ok(const lfpsqp_ctx *c, int NA, int LW) {
  if ((int)c->bnd_host.size() < NA) return false;
  int cnt[32] = {0};
  for (int j = 0; j < NA; j++) if (c->bnd_host[j] != 0.0 && ++cnt[j % LW] > 1) return false;
  return true;
}
}  // namespace

// returns LFPSQP_OK when launched, 1 when this problem shape has no register-resident instantiation (caller falls
// back to the shared-memory warp kernel), < 0 on errors.  LFPSQP_BATCHED_KERNEL=smem forces the fallback (A/B tests);
// LFPSQP_REG_LW selects other instantiations of the C2 shape (A/B measurements, tools/c2_variants.py).
int launch_batched_reg(lfpsqp_ctx *c, BatchedArgs &A) {
  const char *force = getenv("LFPSQP_BATCHED_KERNEL");
  if (force && strcmp(force, "smem") == 0) return 1;
  if (A.prm.linesearch != 0 && !A.prm.disable_linesearch) return 1;   // exact_linesearch! lives in the shared-memory solver
  const int NA = A.n + A.p, ME = A.m + A.p;
  const char *lwenv = getenv("LFPSQP_REG_LW");
  const int lw = lwenv ? atoi(lwenv) : 0;
  switch (A.family) {
    case LFPSQP_FAM_README_INEQ:
      if (ME != 1 || !A.ineq) return 1;
      if (NA <= 32) return launch<SepReadmeIneq, 16, 2, 1, true, false>(c, A);
      if (NA <= 64) {
        if (lw == 32) return launch<SepReadmeIneq, 32, 2, 1, true, false>(c, A);
#ifdef LFPSQP_REG_EXPERIMENTS
        if (lw == 16) return launch<SepReadmeIneq, 16, 4, 1, true, false>(c, A);
        if (NA <= 56 && sparse_ok(c, NA, 8)) {
          if (lw == 82) return launch<SepReadmeIneq, 8, 7, 1, true, true, 128, 2>(c, A);
          if (lw == 83) return launch<SepReadmeIneq, 8, 7, 1, true, true, 128, 3>(c, A);
          if (lw == 84) return launch<SepReadmeIneq, 8, 7, 1, true, true, 160, 2>(c, A);
          if (lw == 85) return launch<SepReadmeIneq, 8, 7, 1, true, true, 96, 4>(c, A);
          if (lw == 86) return launch<SepReadmeIneq, 8, 7, 1, true, true, 128, 4>(c, A);
        }
        if (sparse_ok(c, NA, 16)) {
          if (lw == 163) return launch<SepReadmeIneq, 16, 4, 1, true, true, 128, 3>(c, A);
          if (lw == 164) return launch<SepReadmeIneq, 16, 4, 1, true, true, 128, 4>(c, A);
        }
#endif
        if (NA <= 56 && sparse_ok(c, NA, 8)) return launch<SepReadmeIneq, 8, 7, 1, true, true, 128, 2>(c, A);
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
