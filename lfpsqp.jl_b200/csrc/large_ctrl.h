// large_ctrl.h -- device-resident control block of the large-n mode and the reduction-slot geometry.
#pragma once
#include <stdint.h>

namespace lfpsqp {

constexpr int MAXP = 2048;   // max per-CTA partials per reduction slot
constexpr int NSLOT = 8;

// device-resident control block (one per ctx); mirrored to pinned host memory when the host needs a decision
struct LargeCtrl {
  double s[16];              // generic scalar results (finalize_kernel)
  double rg, dAd, alpha, beta, nr, tol, rpgp, gg, mu, rho, pz, norm_res;
  int iter, lim, status;     // projcg: 0 running, 1 nr<tol, 2 negative curvature, 3 rg<=0, 4 iteration limit
  int pcg_iter, pcg_lim, pcg_status;  // pcg: 0 running, 1 converged (norm_res<=tol), 4 limit
  int rankflag, commfail;    // rankflag: Cholesky pivot below the rank threshold ; commfail: a peer-memory exchange timed out
  double ldiag_min, ldiag_max;   // explicit-inverse guard (large.cu::factorize): estimate of lambda_min(G), trace(G)
  unsigned long long nz_count;   // non-zero entries of the zero-slab map of J (large_gemm.cuh::zero_slab_map_kernel)
  int g_dependent, pad_;         // diagonal blocks of G with a structural non-zero to their left (potf2_inv_indep_kernel); 0 = block diagonal
};

// Peer-memory region every rank exports over CUDA IPC (comm.cu).  First part: pull-model all-reduce kernels of comm.cu
// ([2][PC_MAX + PC_SCAL] doubles, parity double buffer; flags [PC_RANKS][PC_COLS] u64).  Second part (FZ_*): push-model
// mailboxes of the persistent fused projcg kernel (large_fused.cu): 16-byte entries of two self-validating 8-byte words
// {32 value bits, 32-bit exchange number} (NCCL-LL style: 8-byte accesses are atomic, nothing is assumed about 16 bytes),
// one row per source rank; every rank STORES its partial m-vector / scalars into the row [its rank] of every rank's
// region and consumers spin on the entries of their own (local) region.
constexpr int PC_MAX = 8192, PC_SCAL = 32, PC_RANKS = 8, PC_COLS = 16;
constexpr size_t PC_DATA = 2 * (size_t)(PC_MAX + PC_SCAL);
constexpr size_t FZ_OFF = PC_DATA + (size_t)PC_RANKS * PC_COLS;              // doubles from the region start (16-byte aligned)
constexpr size_t FZ_VEC = FZ_OFF;                                           // entries [PC_RANKS][PC_MAX]   (2 doubles each)
constexpr size_t FZ_SCAL = FZ_VEC + 2 * (size_t)PC_RANKS * PC_MAX;          // entries [3 kinds][PC_RANKS]: d.Ad | rp.gp | gp.gp
constexpr size_t FZ_FLAG = FZ_SCAL + 2 * (size_t)PC_RANKS * 4;              // (spare) [PC_RANKS] u64, then this rank's exchange counter (u64)
constexpr size_t FZ_U = (FZ_FLAG + PC_RANKS + 1 + 1) & ~(size_t)1;          // entries [PC_MAX]: the solved u_i, pushed by the rank that owns row i
constexpr size_t PC_REGION_BYTES = (FZ_U + 2 * (size_t)PC_MAX) * 8;
static_assert(FZ_OFF % 2 == 0 && FZ_SCAL % 2 == 0 && FZ_U % 2 == 0, "mailbox entries must be 16-byte aligned");

// bound embedding of the large-n mode (kernels in large_ineq.cuh); device arrays, each nx doubles
struct IneqDev {
  const double *q = nullptr, *r = nullptr, *s = nullptr, *t = nullptr;   // InequalityData (inequality_helper.jl:1-8, :54-82)
  double *Dx = nullptr, *Dy = nullptr, *S = nullptr, *lamy = nullptr;   // inequality_gradient! output, lambda_y
  int64_t nx = 0;
};

// LFPSQP_FAM_SPARSE_QCQP (kernels in large_families.cuh, built by large_spq.cu): device copies of the canonical structures.
// P and the Lagrangian Hessian H = P + sum_i lam_i Qc_i are CSR matrices (32-bit indices); every entry of H lists its sources
// (con -1 = the P entry, else the constraint), P first and then constraints in index order.  The constraints are segments
// (i, r), sorted by i then r: row r of Qc_i merged with Ac[i, r], so that J[i, r] has exactly one owner.
struct SpqDev {
  int64_t n = 0, nh = 0;
  int m = 0, gp = 4, gh = 4;                    // gp / gh: lanes per row of the P / H passes
  const int *prow = nullptr, *pcol = nullptr;
  const double *pval = nullptr, *q = nullptr;
  double r = 0.0;
  const int *hrow = nullptr, *hcol = nullptr, *hsrc_ptr = nullptr, *hsrc_con = nullptr;
  const double *hsrc_val = nullptr;
  double *hval = nullptr;
  const int *con_ptr = nullptr, *seg_row = nullptr, *seg_ptr = nullptr, *seg_col = nullptr;
  const double *seg_a = nullptr, *seg_val = nullptr, *bc = nullptr;
};

// LFPSQP_FAM_SPARSE_QCQP_CSR (kernels in large_spj.cuh, built by large_spq.cu): J kept sparse.  CSR = (SpqDev::con_ptr,
// SpqDev::seg_row, jr); CSC = (cptr, crow, jc), csc_of[s] = CSC slot of segment s.  A row with more than SPJ_CHUNK entries is
// "long": it is cut into chunks of SPJ_CHUNK segments (slots), numbered in row order; row_slot[i] = first slot of row i
// (row_slot[i + 1] == row_slot[i] for a short row), slot_row / slot_beg / slot_end describe slot s, long_row lists the long rows.
constexpr int SPJ_CHUNK = 4096;
struct SpjDev {
  int m = 0, nslot = 0, nlong = 0;
  int64_t nnz = 0;
  const int *cptr = nullptr, *crow = nullptr, *csc_of = nullptr;
  const int *row_slot = nullptr, *slot_row = nullptr, *slot_beg = nullptr, *slot_end = nullptr, *long_row = nullptr;
  double *jr = nullptr, *jc = nullptr;
};

}  // namespace lfpsqp
