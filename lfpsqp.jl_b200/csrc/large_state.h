// large_state.h -- host-side state of the large-n mode (owned by the ctx) and the communicator hooks.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <vector>
#include "../../include/lfpsqp_b200.h"
#include "large_ctrl.h"
#include "ctx.h"

struct LargeState {
  int family = 0;
  int64_t n = 0, n_loc = 0, col0 = 0, ldj = 0, ldm = 0;
  // bound embedding (src/inequality_helper.jl): working vectors are [x-half | y-half], nv = 2 n_loc entries per rank
  bool ineq = false;
  int64_t nv = 0;
  lfpsqp::IneqDev I;
  double *bq = nullptr, *br = nullptr, *bs = nullptr, *bt = nullptr;   // InequalityData (owned copies behind I.q .. I.t)
  double *cvh = nullptr, *cvc = nullptr;   // cvalaug = [h ; c] of ProjPenalty (retractions.jl:29), persistent across calls
  double *pb = nullptr, *Jw = nullptr;     // x-half operand of PJct' v ; J diag(Dy) for the weighted Gram
  lfpsqp::SpqDev spq;                      // LFPSQP_FAM_SPARSE_QCQP: uploaded structures (large_spq.cu)
  // LFPSQP_FAM_SPARSE_QCQP_CSR (family stays LFPSQP_FAM_SPARSE_QCQP, csr set): J in CSR / CSC form instead of S.J
  // (large_spj.cuh); spj_part: chunk partials of the row pass and of jac!'s c, spj_gpart: chunk partial rows of the Gram
  bool csr = false;
  lfpsqp::SpjDev spj;
  double *spj_part = nullptr, *spj_gpart = nullptr;
  int jsplit = 1;                          // row splits a J column pass leaves in cpart: 1 (CSC pass) or nsplit (cols_dot)
  // host-callback family (LFPSQP_FAM_HOST): the callbacks, pinned staging buffers, device staging of Jc (n x m)
  lfpsqp_host_callbacks cb = {};
  double *hx = nullptr, *hv = nullptr, *hw = nullptr, *hlam = nullptr, *hc = nullptr, *hJ = nullptr, *Jstage = nullptr;
  int cb_err = 0;
  // persistent fused projcg (large_fused.cu)
  bool fused_ok = false;
  int fused_grid = 0;
  double *fused_part = nullptr;
  double *Ginv = nullptr;                  // explicit G^-1 = L^-T L^-1 (m x m, symmetric) for the one-phase solve of the fused kernel
  // explicit-inverse guard: u = G^-1 t loses cond(G) eps, two triangular solves only cond(L) eps.  factorize() bounds cond(G)
  // from above by kappa = trace(G) * lambda_max(G^-1) (power iterations on the explicit inverse); above `inverse_guard` the
  // fused kernel runs the two triangular phases instead.  force_inverse: LFPSQP_EXPLICIT_INVERSE=0/1 at setup forces either path
  // (tests), -1 leaves the choice to the guard
  // rank-deficient Jacobians (large_eig.cu): after a failed Cholesky pivot test the solves use the truncated pseudo-inverse
  // G^+ (held in Ginv) of the eigen-decomposed Gram; rank_cur feeds projcg's iteration cap and the NR / ProjPenalty choice
  bool pinv_active = false, prefer_pinv = false;
  int rank_cur = 0;
  double *eigV = nullptr, *eigT = nullptr, *eigLam = nullptr;
  unsigned long long *eigScratch = nullptr;    // [32] convergence per sweep | barrier counter | sweeps done
  double *noise_dev = nullptr; size_t noise_cap = 0; int64_t noise_T = 0;   // caller-supplied noise rows (lfpsqp_ctx_set_noise), beta > 0
  bool explicit_inverse_ok = true, guard_pending = false;
  int force_inverse = -1;
  double inverse_guard = 1e6, pivot_ratio2 = 1.0;   // pivot_ratio2: the last kappa
  int m = 0, sm_count = 148, world = 1, rank = 0;
  cudaStream_t stream = nullptr;
  lfpsqp_params prm;
  CommState *comm = nullptr;
  // family parameters (device)
  const double *p_Q = nullptr, *p_A = nullptr, *p_b = nullptr, *p_xt = nullptr, *p_w = nullptr;
  // matrices
  double *J = nullptr, *G = nullptr, *XT = nullptr, *Linv = nullptr, *Dblk = nullptr, *tmp64 = nullptr, *thresh = nullptr,
         *gemm_ws = nullptr, *Dnr = nullptr, *pairws = nullptr;
  size_t gemm_ws_bytes = 0;
  // zero-slab map of J for the Gram (large_gemm.cuh): J is stored dense, but the SYRK skips K chunks in which the rows of a tile
  // are all zero.  gram_mode 0: not decided (scan + skipping kernel, density read with the next control block), 1: block-sparse
  // (keep scanning: values may change), 2: dense (plain kernel, no scan; sticky -- zeros appearing later only cost time)
  // g_blockdiag: the previous factorisation found G block diagonal (every diagonal block independent) -> the next one reads the
  // count back right after the parallel diagonal factorisation and, if it is still 0, enqueues neither the Cholesky chain nor the
  // inverse's GEMM levels (hundreds of launches that would all return at once)
  // gram_skip: structure detection (zero-slab map, block flags) is on; LFPSQP_GRAM_SKIP=0 at setup turns it off (tests compare
  // against the plain dense path bit for bit)
  int g_blockdiag = 0;
  bool gdep_pending = false, gram_skip = true;
  int *invflag = nullptr;      // [nblk][nblk] block structure of L^-1 (scanned after the inverse) for the triangular passes; null: off
  bool invflag_valid = false;
  int *blkflag = nullptr;      // [nblk][nblk] block structure of G / L for the factorisation (large_gemm.cuh::GemmExt::bf)
  unsigned char *nzmap = nullptr;
  int64_t nz_ld = 0;
  int nz_rows = 0, gram_mode = 0, max_dyn_smem = 48 * 1024;
  bool nz_pending = false;
  bool jmap_valid = false;   // nzmap describes the CURRENT contents of S.J (scanned by the last Gram, J not rewritten since): the
                             // unfused passes over J (rows_dot / cols_dot) skip its all-zero slabs too
  // n_loc vectors
  double *x = nullptr, *xnew = nullptr, *xtil = nullptr, *g = nullptr, *d = nullptr, *nd = nullptr, *w0 = nullptr,
         *w1 = nullptr, *w2 = nullptr, *w3 = nullptr, *w4 = nullptr, *hdiag = nullptr, *ex[4] = {nullptr, nullptr, nullptr, nullptr};
  // m vectors (replicated on every rank)
  double *cval = nullptr, *lam = nullptr, *tm = nullptr, *ty = nullptr, *tu = nullptr, *nr_t1 = nullptr, *nr_t2 = nullptr,
         *nr_dc = nullptr;
  double *xfull = nullptr, *xfull_h = nullptr, *vfull = nullptr;   // THOMSON column-sharded: all-gathered coordinates (scratch / Hessian point / direction)
  double *cpart = nullptr;   // pass-2 partial column sums [nsplit][n_loc]
  int nsplit = 1, rows_per_split = 1;
  double *lp = nullptr, *gpart = nullptr, *commbuf = nullptr;   // loop partials, generic partials [NSLOT][MAXP]
  lfpsqp::LargeCtrl *ctrl = nullptr, *hctrl = nullptr;
  int vgrid = 1, np_loop = 1, np_loop_raw = 1, cg_chunk = 2, pcg_chunk = 2;
  cudaEvent_t ev_g0 = nullptr, ev_g1 = nullptr;
  cudaStream_t side_stream = nullptr;                  // look-ahead of the blocked Cholesky (large.cu::factorize)
  cudaEvent_t ev_panel = nullptr, ev_potf = nullptr;
  std::vector<void *> owned;
  // lfpsqp_large_last_dispatch: what the last large-n entry call enqueued, recorded on the host where the launches are made and
  // cleared by every entry call (LARGE_DISP_* below).  disp_syrk: the product being enqueued is the Gram's SYRK.
  int64_t disp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  bool disp_syrk = false;
  // counters
  int64_t collectives = 0, launches = 0, projcg_iters = 0, projcg_negcurv = 0, armijo_trials = 0, retract_outer = 0, retract_pcg = 0,
          pp_backtracks = 0, newton_accepted = 0, factorizations = 0, f_evals = 0;
  double ms_factor = 0, ms_projcg = 0, ms_linesearch = 0, t_factor_pending = 0;
  void reset_counters() {
    ms_factor = ms_projcg = ms_linesearch = t_factor_pending = 0;
    launches = projcg_iters = projcg_negcurv = armijo_trials = retract_outer = retract_pcg = pp_backtracks = 0;
    newton_accepted = factorizations = f_evals = 0;
  }
};

// entries of LargeState::disp (the layout of lfpsqp_large_last_dispatch, include/lfpsqp_b200.h)
enum {
  LARGE_DISP_GEMM = 0,          // mask of dgemm_nt instantiations
  LARGE_DISP_KSPLIT_GRID = 1,   // largest split-K factor of a product with too few tiles for the GPU (0: none)
  LARGE_DISP_KSPLIT_WAVE = 2,   // largest wave-quantisation split-K factor of a SYRK (0: none)
  LARGE_DISP_ROWS_DOT = 3,      // mask of rows_dot_kernel instantiations
  LARGE_DISP_FUSED_SINGLE = 4,  // launches of the single-GPU explicit-inverse fused projcg kernel (fused_projcg_kernel<false, false>)
  LARGE_DISP_FUSED_GENERAL = 5, // launches of the other fused projcg instantiations (column-sharded or triangular solve)
  LARGE_DISP_FUSED_PCG = 6,     // launches of the fused pcg! kernel
  LARGE_DISP_SOLVE = 7,         // mask of the forms u = G^-1 t was applied in
};
enum { LARGE_SOLVE_EXPLICIT = 1, LARGE_SOLVE_TRIANGULAR = 2, LARGE_SOLVE_PINV = 4 };
// the solve form of a fused kernel that applies S.Ginv: G^-1, or G^+ once the factorisation lost rank (large.cu::factorize_pinv)
inline int64_t large_ginv_form(const LargeState &S) { return S.pinv_active ? LARGE_SOLVE_PINV : LARGE_SOLVE_EXPLICIT; }

// large_fused.cu: one cooperative kernel per chunk of projcg iterations (returns 1 when not eligible -> unfused path)
int fused_projcg_chunk(LargeState &S, int iters, int first, double *xs, double *r, double *dc, double *Ad, double *rp, double *gp);
int fused_pcg(LargeState &S, double *dx, double *r, double *pv, double *z);   // the whole pcg! call as one launch
void fused_projcg_init(LargeState &S, int device);

// large_spq.cu: LFPSQP_FAM_SPARSE_QCQP.  spq_build validates the descriptor (LFPSQP_ERR_ARG with a message) and builds the
// canonical host form; spq_upload copies it into S.spq (false: allocation or copy failed)
struct SpqHost {
  int64_t n = 0;
  int m = 0;
  double r = 0.0;
  std::vector<double> q, bc, pval, hsrc_val, seg_a, seg_val;
  std::vector<int> prow, pcol, hrow, hcol, hsrc_ptr, hsrc_con, con_ptr, seg_row, seg_ptr, seg_col;
};
int spq_build(lfpsqp_ctx *c, const lfpsqp_sparse_qcqp *D, int64_t n, int64_t m, SpqHost &H);
bool spq_upload(LargeState &S, const SpqHost &H);
// LFPSQP_FAM_SPARSE_QCQP_CSR: the CSC pattern of J and the chunk partition of long rows (host, fixed order), the two value
// arrays and the chunk partial buffers -> S.spj, S.spj_part, S.spj_gpart (false: allocation or copy failed)
bool spj_upload(LargeState &S, const SpqHost &H);

// large_eig.cu: eigen-decomposition of the Gram (one-sided Jacobi) -> scaled eigenvectors for the pseudo-inverse
int large_eig_pinv_factors(LargeState &S, double *G, double *Vt, double *lam, int lower_only, int *sweeps_dev, unsigned long long *conv_dev,
                           unsigned *bar_dev);

// comm.cu
void comm_allreduce(LargeState &S, double *buf, size_t count);                  // in-place sum over ranks
void comm_allreduce_scalars(LargeState &S, unsigned summask, unsigned maxmask); // ctrl->s[k] for the masked slots
void comm_allreduce_loop_slot(LargeState &S, int slot, int np);                 // lp[slot][0] = sum over ranks of sum_i lp[slot][i]
void comm_allreduce_loop_slots_cg(LargeState &S, int par);                      // slots 1 and 2+par
void comm_release(LargeState &S);
