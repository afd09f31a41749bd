// large.cu -- large-n mode: one instance, dense J (m x n) column-sharded over the ranks, host-orchestrated.
//
// The reference's driver (src/optimize.jl:119-443) runs here on the host as stream orchestration; every O(n) /
// O(mn) / O(m^2 n) operation is a hand-written kernel (large_gemm.cuh, large_kernels.cuh, large_families.cuh).
// Inner loops (projcg!, pcg!) are device-predicated: their kernels test ctrl->status, so iterations are enqueued
// in chunks and the host reads the control block once per chunk.
// Finite bounds run the reference's 2n-variable embedding (src/inequality_helper.jl): working vectors become
// [x-half | y-half] and the operators take the closed forms of large_ineq.cuh.  LFPSQP_FAM_HOST evaluates f / grad! /
// c! / jac! / hess_lag_vec! through host callbacks (the explicit-derivative core, optimize.jl:119): generic problems.
#include <cuda_runtime.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <chrono>
#include <vector>

#include "ctx.h"
#include "large_gemm.cuh"
#include "large_kernels.cuh"
#include "large_families.cuh"
#include "large_ineq.cuh"
#include "large_spj.cuh"
#include "large_state.h"

using namespace lfpsqp;

#define CK(call)                                                        \
  do {                                                                  \
    cudaError_t e__ = (call);                                           \
    if (e__ != cudaSuccess) return c->cuda_fail(e__, #call);            \
  } while (0)

static inline int64_t up2(int64_t v) { return (v + 1) & ~(int64_t)1; }
static inline double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ------------------------------------------------------------------ small launch helpers
template <class F>
static void vec(LargeState &S, int64_t n, F f, int s0 = 0, int nsum = 0, int domax = 0) {
  vec_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, f, S.gpart, s0, nsum, domax);
}
// repmask: slots computed from REPLICATED m-vectors (identical on every rank) -- not all-reduced
static void finalize(LargeState &S, unsigned summask, unsigned maxmask, unsigned repmask = 0) {
  finalize_kernel<<<1, 256, 0, S.stream>>>(S.gpart, S.vgrid, summask, maxmask, S.ctrl);
  S.launches++;
  if (S.world > 1 && ((summask | maxmask) & ~repmask)) comm_allreduce_scalars(S, summask & ~repmask, maxmask & ~repmask);
}
static int read_ctrl(lfpsqp_ctx *c, LargeState &S) {
  CK(cudaMemcpyAsync(S.hctrl, S.ctrl, sizeof(LargeCtrl), cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  CK(cudaGetLastError());   // a refused launch (bad configuration) since the last check must not pass silently
  if (S.hctrl->commfail) return c->fail(LFPSQP_ERR_COMM, "a peer-memory exchange of the column-sharded mode timed out (a rank died or fell > 4 s behind)");
  if (S.gdep_pending) { S.gdep_pending = false; S.g_blockdiag = (S.hctrl->g_dependent == 0) ? 1 : 0; }
  if (S.nz_pending) {       // density of the zero-slab map of J -> keep skipping (block-sparse J) or use the plain SYRK from now on
    S.nz_pending = false;
    // out of the (64-row slab, K chunk) pairs the scan visits; nz_ld is padded past the last chunk and does not count
    const double total = (double)S.nz_rows * (double)std::max<int64_t>((S.n_loc + GM_BK - 1) / GM_BK, 1);
    S.gram_mode = ((double)S.hctrl->nz_count > 0.5 * total) ? 2 : 1;
  }
  if (S.guard_pending) {    // pivots of the factor just computed -> which solve the fused projcg kernel may use
    S.guard_pending = false;
    const double lo = S.hctrl->ldiag_min, hi = S.hctrl->ldiag_max;   // ~lambda_min(G) (from above), trace(G)
    S.pivot_ratio2 = (lo > 0.0) ? hi / lo : INFINITY;
    S.explicit_inverse_ok = S.force_inverse >= 0 ? S.force_inverse == 1 : S.pivot_ratio2 <= S.inverse_guard;
  }
  return 0;
}
static void write_ctrl_fields(LargeState &S) {  // push the host copy (tolerances, limits, statuses) to the device
  cudaMemcpyAsync(S.ctrl, S.hctrl, sizeof(LargeCtrl), cudaMemcpyHostToDevice, S.stream);
}
static void reset_ctrl(LargeState &S) {   // a cleared control block on the host and the device
  memset(S.hctrl, 0, sizeof(LargeCtrl));
  write_ctrl_fields(S);
}

// lfpsqp_large_last_dispatch bits of a dgemm_nt instantiation: 1 <128> lean, 2 <128> with the extras' prologue, 4 <64>,
// 8 <128, SKIP>; bits 0-3 for the Gram's SYRK, bits 4-7 for every other product
static void note_gemm(LargeState &S, int bit) { S.disp[LARGE_DISP_GEMM] |= (int64_t)bit << (S.disp_syrk ? 0 : 4); }

// C (op)= A B' with optional split-K through S.gemm_ws
static void gemm_nt(LargeState &S, int M, int N, int K, const double *A, int64_t lda, const double *B, int64_t ldb, double *C,
                    int64_t ldc, int mode, int lower, const GemmExt *ext = nullptr) {
  if (M <= 0 || N <= 0) return;
  const bool narrow = (N <= 64);
  const int BN = narrow ? 64 : 128;
  dim3 grid((N + BN - 1) / BN, (M + GM_BM - 1) / GM_BM, 1);
  int tiles = grid.x * grid.y;
  if (lower) tiles = (tiles + grid.y) / 2;
  int ksplit = 1;
  GemmExt X; if (ext) X = *ext;
  if (X.batch > 1) {   // independent products of one shape: blockIdx.z = product
    grid.z = X.batch;
  } else if (mode != GEMM_SUB && tiles * 2 <= S.sm_count && K >= 1024 && !X.tri) {
    ksplit = std::min(std::min(16, S.sm_count / tiles), K / 256);
    while (ksplit > 1 && (size_t)ksplit * M * (N + 1) * 8 > S.gemm_ws_bytes) ksplit--;
    if (ksplit < 1) ksplit = 1;
    if (ksplit > 1) S.disp[LARGE_DISP_KSPLIT_GRID] = std::max<int64_t>(S.disp[LARGE_DISP_KSPLIT_GRID], ksplit);
  } else if (mode == GEMM_ASSIGN && lower && K >= 8192 && tiles < S.sm_count) {
    // wave quantisation of a SYRK that does not fill one wave (C5: 136 lower tiles on 148 SMs = 92 %): split K so that
    // tiles x ksplit fills whole waves (C5: 13 -> 1768 CTAs = 11.95 waves; measured 27.2 -> 28.9 TFLOP/s).  With several
    // waves already (C4: 528 tiles) the split measured slower (7.6 -> 8.7 ms): not applied.
    auto eff = [&](int ks) { int64_t w = (int64_t)tiles * ks; return (double)w / (double)(((w + S.sm_count - 1) / S.sm_count) * S.sm_count); };
    int best = 1;
    for (int ks = 2; ks <= 16; ks++) {
      if ((size_t)ks * M * (N + 1) * 8 > S.gemm_ws_bytes || K / ks < 2048) break;
      if (eff(ks) > eff(best) + 0.02) best = ks;
    }
    ksplit = best;
    if (ksplit > 1) S.disp[LARGE_DISP_KSPLIT_WAVE] = std::max<int64_t>(S.disp[LARGE_DISP_KSPLIT_WAVE], ksplit);
  }
  // zero-slab skipping (SYRK of a block-sparse J): the chunk list of one K slice must fit behind the tiles in shared memory
  const int kchunks = (K + GM_BK - 1) / GM_BK, per = (kchunks + ksplit - 1) / ksplit;
  const size_t skip_smem = dgemm_smem_bytes<128>() + (size_t)per * sizeof(int);
  const bool skip = X.nz && X.batch <= 1 && !narrow && skip_smem <= (size_t)S.max_dyn_smem;
  const bool lean = !ext;   // plain product: the instantiation without the extras' prologue
  note_gemm(S, skip ? 8 : narrow ? 4 : lean ? 1 : 2);
  const auto kern = skip ? dgemm_nt_kernel<128, true> : narrow ? dgemm_nt_kernel<64> : lean ? dgemm_nt_kernel<128, false, false> : dgemm_nt_kernel<128>;
  const size_t smem = skip ? skip_smem : narrow ? dgemm_smem_bytes<64>() : dgemm_smem_bytes<128>();
  if (ksplit == 1) {
    kern<<<grid, 256, smem, S.stream>>>(M, N, K, A, lda, B, ldb, C, ldc, mode, lower, 1, 0, X);
    S.launches++;
  } else {
    grid.z = ksplit;
    const int64_t ldw = (N + 1) & ~1;   // even row pitch: the epilogue stores 16-byte pairs
    const int64_t stride = (int64_t)M * ldw;
    kern<<<grid, 256, smem, S.stream>>>(M, N, K, A, lda, B, ldb, S.gemm_ws, ldw, GEMM_ASSIGN, lower, ksplit, stride, X);
    const double *ws = S.gemm_ws;
    const double sgn = (mode == GEMM_ASSIGN_NEG) ? -1.0 : 1.0;
    const int lo = lower;
    vec(S, (int64_t)M * N, [=] __device__(int64_t e0, double *) {
      int r = (int)(e0 / N), cc = (int)(e0 % N);
      if (lo && (r / GM_BM) * GM_BM + GM_BM <= (cc / BN) * BN) return;   // tile was skipped
      const int64_t e = (int64_t)r * ldw + cc;
      double s = 0.0;
      for (int z = 0; z < ksplit; z++) s += ws[(int64_t)z * stride + e];
      C[(int64_t)r * ldc + cc] = sgn * s;
    });
    S.launches += 2;
  }
}

static void rows_dot(LargeState &S, const double *Jm, int64_t ld, int m, int64_t ncols, const double *v, double *t, int pred) {
  if (m <= 0) return;
  const bool skip = Jm == S.J && S.jmap_valid && S.gram_mode == 1;   // block-sparse J: same pass, loads of all-zero slabs not issued
  const int R = m >= 8 * S.sm_count ? 4 : m >= 2 * S.sm_count ? 2 : 1;
  static decltype(&rows_dot_kernel<1>) const kern[2][3] = {{rows_dot_kernel<1>, rows_dot_kernel<2>, rows_dot_kernel<4>},
                                                           {rows_dot_kernel<1, true>, rows_dot_kernel<2, true>, rows_dot_kernel<4, true>}};
  kern[skip][R / 2]<<<(m + R - 1) / R, 256, 0, S.stream>>>(Jm, ld, m, ncols, v, t, S.ctrl, pred, skip ? S.nzmap : nullptr, skip ? S.nz_ld : 0);
  S.disp[LARGE_DISP_ROWS_DOT] |= R << (skip ? 3 : 0);   // bits 0-2: R = 1, 2, 4 ; 3-5: SKIP
  S.launches++;
}
static void cols_dot(LargeState &S, const double *Jm, int64_t ld, int m, int64_t ncols, const double *u, int pred) {
  if (m <= 0) return;
  dim3 grid((unsigned)((ncols + 511) / 512), S.nsplit);
  if (Jm == S.J && S.jmap_valid && S.gram_mode == 1)
    cols_dot_kernel<true><<<grid, 256, S.rows_per_split * sizeof(double), S.stream>>>(Jm, ld, m, ncols, u, S.cpart, S.rows_per_split, S.ctrl, pred, S.nzmap, S.nz_ld);
  else
    cols_dot_kernel<false><<<grid, 256, S.rows_per_split * sizeof(double), S.stream>>>(Jm, ld, m, ncols, u, S.cpart, S.rows_per_split, S.ctrl, pred);
  S.launches++;
}

// ---- the passes over the constraint Jacobian: dense S.J (rows_dot / cols_dot) or, for LFPSQP_FAM_SPARSE_QCQP_CSR, its CSR /
// CSC value arrays (large_spj.cuh).  jcols leaves S.jsplit row splits in S.cpart.
static int spj_items_grid(const LargeState &S) { return (int)(((int64_t)S.m + S.spj.nslot + 7) / 8); }   // one warp per item
static void jrows(LargeState &S, const double *v, double *t, int pred) {   // t = J v (first n_loc entries of v)
  if (!S.csr) { rows_dot(S, S.J, S.ldj, S.m, S.n_loc, v, t, pred); return; }
  if (S.m <= 0) return;
  spj_rows_kernel<<<spj_items_grid(S), 256, 0, S.stream>>>(S.spj, S.spq.con_ptr, S.spq.seg_row, v, t, S.spj_part, S.ctrl, pred);
  S.launches++;
  if (S.spj.nlong > 0) {
    spj_combine_kernel<<<(S.spj.nlong + 255) / 256, 256, 0, S.stream>>>(S.spj, S.spj_part, nullptr, t, S.ctrl, pred);
    S.launches++;
  }
  S.disp[LARGE_DISP_ROWS_DOT] |= 64;
}
static void jcols(LargeState &S, const double *u, int pred) {   // S.cpart = J'u
  if (!S.csr) { cols_dot(S, S.J, S.ldj, S.m, S.n_loc, u, pred); return; }
  if (S.m <= 0) return;
  spj_cols_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.spj, S.n_loc, u, S.cpart, S.ctrl, pred);
  S.launches++;
  S.disp[LARGE_DISP_ROWS_DOT] |= 128;
}
// jac! of the CSR form: cval = c(x), with jac also both value arrays of J
static void spj_cjac(LargeState &S, bool jac, double *cval, const double *x) {
  const lfpsqp::SpqDev &D = S.spq;
  if (jac) spj_cjac_kernel<true><<<spj_items_grid(S), 256, 0, S.stream>>>(S.spj, D.con_ptr, D.seg_row, D.seg_a, D.seg_ptr, D.seg_col, D.seg_val, D.bc, x, cval, S.spj_part);
  else spj_cjac_kernel<false><<<spj_items_grid(S), 256, 0, S.stream>>>(S.spj, D.con_ptr, D.seg_row, D.seg_a, D.seg_ptr, D.seg_col, D.seg_val, D.bc, x, cval, S.spj_part);
  S.launches++;
  if (S.spj.nlong > 0) {
    spj_combine_kernel<<<(S.spj.nlong + 255) / 256, 256, 0, S.stream>>>(S.spj, S.spj_part, D.bc, cval, S.ctrl, 0);
    S.launches++;
  }
}
// S.G (lower triangle, every entry written) = J J', or J diag(Dy^2) J' with bounds, over the sparsity pattern
static void spj_gram(LargeState &S) {
  const int m = S.m;
  const size_t smem = (size_t)m * sizeof(double);
  const unsigned grid = (unsigned)(m + S.spj.nslot);
  const lfpsqp::SpqDev &D = S.spq;
  if (S.ineq) spj_gram_kernel<true><<<grid, 32, smem, S.stream>>>(S.spj, D.con_ptr, D.seg_row, S.I.Dy, S.G, S.ldm, S.spj_gpart);
  else spj_gram_kernel<false><<<grid, 32, smem, S.stream>>>(S.spj, D.con_ptr, D.seg_row, nullptr, S.G, S.ldm, S.spj_gpart);
  S.launches++;
  if (S.spj.nlong > 0) {
    spj_gram_combine_kernel<<<dim3((unsigned)((m + 255) / 256), (unsigned)S.spj.nlong), 256, 0, S.stream>>>(S.spj, S.spj_gpart, S.G, S.ldm);
    S.launches++;
  }
  S.disp[LARGE_DISP_GEMM] |= 256;
}
// u = T t with T = L^-1 (lower) or T = L^-T (upper, S.XT) of the cached factor; u_copy (optional) receives u as well
static void tri_gemv(LargeState &S, int upper, const double *t, double *u, double *u_copy, int pred) {
  const int m = S.m;
  tri_gemv_kernel<<<(m + 7) / 8, 256, m * sizeof(double), S.stream>>>(upper ? S.XT : S.Linv, S.ldm, m, t, u, upper, u_copy, S.ctrl, pred,
                                                                      S.invflag_valid ? S.invflag : nullptr, S.nz_rows);
  S.launches++;
}
// u = (J J')^-1 t through the cached factor: y = L^-1 t ; u = L^-T y
static void gram_solve(LargeState &S, const double *t, double *u, double *u_copy, int pred) {
  const int m = S.m;
  if (S.pinv_active) {   // rank-deficient: u = G^+ t (one dense m x m pass; optimize.jl:297-302 equivalent, large_eig.cu)
    rows_dot(S, S.Ginv, S.ldm, m, m, t, u, pred);
    S.disp[LARGE_DISP_SOLVE] |= LARGE_SOLVE_PINV;
    if (u_copy) vec(S, m, [=] __device__(int64_t a, double *) { u_copy[a] = u[a]; });
    S.launches++;
    return;
  }
  tri_gemv(S, 0, t, S.ty, nullptr, pred);
  tri_gemv(S, 1, S.ty, u, u_copy, pred);
  S.disp[LARGE_DISP_SOLVE] |= LARGE_SOLVE_TRIANGULAR;
}

// ------------------------------------------------------------------ family dispatch (device callbacks, whole-GPU kernels)
static void thomson_grid(LargeState &S, int npl, dim3 &grid) {   // npl = owned points
  int ib = (npl + 255) / 256;
  int js = std::max(1, std::min(16, (2 * S.sm_count) / ib));
  grid = dim3(ib, js);
}
// Thomson's callbacks need the coordinates of ALL points (SURVEY.md 8e-iv): all-gather of this rank's entries of an n-vector,
// done as an all-reduce of the zero-padded vector (98 KB at N = 4096).  Single GPU: the vector itself.
static const double *thomson_gather(LargeState &S, const double *v_loc, double *full) {
  if (S.world <= 1) return v_loc;
  cudaMemsetAsync(full, 0, (size_t)S.n * sizeof(double), S.stream);
  cudaMemcpyAsync(full + S.col0, v_loc, (size_t)S.n_loc * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);
  comm_allreduce(S, full, (size_t)S.n);
  return full;
}
// ---- host-callback family: the first n entries of a device vector -> pinned S.hx (blocking; also orders every earlier
// H2D copy out of the pinned staging buffers before the callback may overwrite them)
static void host_x(LargeState &S, const double *x) {
  cudaMemcpyAsync(S.hx, x, S.n_loc * sizeof(double), cudaMemcpyDeviceToHost, S.stream);
  cudaStreamSynchronize(S.stream);
}
__global__ void set_partials_kernel(double *part, int np, double v) {
  for (int i = threadIdx.x; i < np; i += blockDim.x) part[i] = (i == 0) ? v : 0.0;
}
// SPARSE_QCQP CSR passes (spq_csr_kernel): mode 0 f partials, 1 grad, 2 Hessian action; G lanes per row from setup
static void spq_csr(LargeState &S, int mode, const int *rp, const int *ci, const double *v, int lanes, const double *x, double *y,
                    double *part, int pred) {
  const lfpsqp::SpqDev &D = S.spq;
  const int64_t n = D.n;
#define SPQ_CSR(G, M) spq_csr_kernel<G, M><<<S.vgrid, 256, 0, S.stream>>>(n, rp, ci, v, x, D.q, D.r, y, part, S.ctrl, pred)
  if (lanes == 32) { if (mode == 0) SPQ_CSR(32, 0); else if (mode == 1) SPQ_CSR(32, 1); else SPQ_CSR(32, 2); }
  else { if (mode == 0) SPQ_CSR(4, 0); else if (mode == 1) SPQ_CSR(4, 1); else SPQ_CSR(4, 2); }
#undef SPQ_CSR
}
static void fam_f(LargeState &S, const double *x) {  // -> gpart slot 0 (sum); caller finalizes s[0]
  if (S.family == LFPSQP_FAM_HOST) {
    host_x(S, x);
    double fv = NAN;
    if (S.cb.f(S.cb.user, S.hx, S.n, &fv)) S.cb_err = 1;
    set_partials_kernel<<<1, 256, 0, S.stream>>>(S.gpart, S.vgrid, fv);
  } else if (S.family == LFPSQP_FAM_DIAGQUAD) {
    const double *xt = S.p_xt, *w = S.p_w;
    vec(S, S.n_loc, [=] __device__(int64_t j, double *acc) { double t = x[j] - xt[j]; acc[0] += 0.5 * w[j] * t * t; }, 0, 1);
  } else if (S.family == LFPSQP_FAM_SPARSE_QCQP) {
    spq_csr(S, 0, S.spq.prow, S.spq.pcol, S.spq.pval, S.spq.gp, x, nullptr, S.gpart, 0);
  } else {
    const int np = (int)(S.n / 3), npl = (int)(S.n_loc / 3), i0 = (int)(S.col0 / 3);
    const double *xf = thomson_gather(S, x, S.xfull);
    dim3 grid; thomson_grid(S, npl, grid);
    thomson_pair_kernel<0><<<grid, 256, 0, S.stream>>>(np, i0, npl, xf, nullptr, nullptr, S.gpart, 0, S.ctrl, 0);
    // the pair kernel wrote grid.x*grid.y partials: fold them into the vgrid partials finalize() expects
    collapse_partials_kernel<<<1, 256, 0, S.stream>>>(S.gpart, grid.x * grid.y, S.vgrid);
  }
  S.launches++; S.f_evals++;
}
static void fam_grad(LargeState &S, double *g, const double *x) {
  if (S.family == LFPSQP_FAM_HOST) {
    host_x(S, x);
    if (S.cb.grad(S.cb.user, S.hv, S.hx, S.n)) S.cb_err = 1;
    cudaMemcpyAsync(g, S.hv, S.n_loc * sizeof(double), cudaMemcpyHostToDevice, S.stream);
  } else if (S.family == LFPSQP_FAM_DIAGQUAD) {
    const double *xt = S.p_xt, *w = S.p_w;
    vec(S, S.n_loc, [=] __device__(int64_t j, double *) { g[j] = w[j] * (x[j] - xt[j]); });
  } else if (S.family == LFPSQP_FAM_SPARSE_QCQP) {
    spq_csr(S, 1, S.spq.prow, S.spq.pcol, S.spq.pval, S.spq.gp, x, g, nullptr, 0);
  } else {
    const int np = (int)(S.n / 3), npl = (int)(S.n_loc / 3), i0 = (int)(S.col0 / 3);
    const double *xf = thomson_gather(S, x, S.xfull);
    dim3 grid; thomson_grid(S, npl, grid);
    thomson_pair_kernel<1><<<grid, 256, 0, S.stream>>>(np, i0, npl, xf, nullptr, S.pairws, nullptr, 0, S.ctrl, 0);
    thomson_reduce_kernel<1><<<(3 * npl + 255) / 256, 256, 0, S.stream>>>(npl, grid.y, S.pairws, nullptr, nullptr, g, nullptr, 0, S.ctrl, 0);
    S.launches++;
  }
  S.launches++;
}
// cval = c(x); with jac also the Jacobian (jac! writes both, autodiff_generators.jl:40-42)
static void fam_c_jac(LargeState &S, bool jac, double *cval, const double *x) {
  double *Jout = jac ? S.J : nullptr;
  // J is rewritten: its zero-slab map is stale until the next Gram scans it -- except for THOMSON, whose jac! kernel writes the
  // same three structural entries of every row whatever x is (a map entry can then only be conservatively non-zero)
  if (jac && S.family != LFPSQP_FAM_THOMSON) S.jmap_valid = false;
  const int m = S.m;
  if (S.family == LFPSQP_FAM_HOST) {
    host_x(S, x);
    if (Jout) {  // jac!(Jc, cval, x): Jc is m x n column-major (optimize.jl:189) = n x m row-major -> transposed into J (= Jct)
      if (S.cb.jac(S.cb.user, S.hJ, S.hc, S.hx, S.n, m)) S.cb_err = 1;
      cudaMemcpyAsync(S.Jstage, S.hJ, (size_t)m * S.n_loc * sizeof(double), cudaMemcpyHostToDevice, S.stream);
      dim3 tg((m + 31) / 32, (unsigned)((S.n_loc + 31) / 32));
      transpose_kernel<<<tg, 256, 0, S.stream>>>(S.Jstage, m, Jout, S.ldj, (int)S.n_loc, m);
    } else if (S.cb.c(S.cb.user, S.hc, S.hx, S.n, m)) S.cb_err = 1;
    cudaMemcpyAsync(cval, S.hc, (size_t)m * sizeof(double), cudaMemcpyHostToDevice, S.stream);
    S.launches++;
  } else if (S.family == LFPSQP_FAM_DIAGQUAD) {
    if (Jout) dq_rows_kernel<2, true><<<(m + 1) / 2, 256, 0, S.stream>>>(S.p_Q, S.p_A, S.ldj, m, S.n_loc, x, Jout, cval);
    else dq_rows_kernel<2, false><<<(m + 1) / 2, 256, 0, S.stream>>>(S.p_Q, S.p_A, S.ldj, m, S.n_loc, x, nullptr, cval);
    if (S.world > 1) comm_allreduce(S, cval, m);
    const double *b = S.p_b;
    vec(S, m, [=] __device__(int64_t i, double *) { cval[i] -= b[i]; });
    S.launches += 2;
  } else if (S.family == LFPSQP_FAM_SPARSE_QCQP) {
    if (m <= 0) return;
    const lfpsqp::SpqDev &D = S.spq;
    if (S.csr) { spj_cjac(S, jac, cval, x); return; }
    if (Jout) spq_cjac_kernel<true><<<m, 256, 0, S.stream>>>(D.con_ptr, D.seg_row, D.seg_a, D.seg_ptr, D.seg_col, D.seg_val, D.bc, x, Jout, S.ldj, cval);
    else spq_cjac_kernel<false><<<m, 256, 0, S.stream>>>(D.con_ptr, D.seg_row, D.seg_a, D.seg_ptr, D.seg_col, D.seg_val, D.bc, x, nullptr, S.ldj, cval);
    S.launches++;
  } else {
    if (Jout) cudaMemsetAsync(Jout, 0, (size_t)m * S.ldj * sizeof(double), S.stream);  // dense-treated, as the reference
    const int npl = (int)(S.n_loc / 3), i0 = (int)(S.col0 / 3);
    if (S.world > 1) cudaMemsetAsync(cval, 0, (size_t)m * sizeof(double), S.stream);    // the other ranks' rows: summed in below
    thomson_c_kernel<<<(npl + 255) / 256, 256, 0, S.stream>>>(npl, i0, x, cval, Jout, S.ldj);
    if (S.world > 1) comm_allreduce(S, cval, m);
    S.launches += 2;
  }
}
// per outer iteration: whatever of the Lagrangian Hessian depends only on (x, lambda)
static void fam_hess_prepare(LargeState &S, const double *x, const double *lam) {
  if (S.family == LFPSQP_FAM_THOMSON) {  // all-gathered coordinates of the point the Hessian is taken at (once per outer iteration)
    if (S.world > 1) thomson_gather(S, x, S.xfull_h);
  } else if (S.family == LFPSQP_FAM_HOST) {  // the closure of optimize.jl:227-231 reads the current x and lambda: cache them on the host
    host_x(S, x);
    if (S.m > 0) { cudaMemcpyAsync(S.hlam, lam, S.m * sizeof(double), cudaMemcpyDeviceToHost, S.stream); cudaStreamSynchronize(S.stream); }
  } else if (S.family == LFPSQP_FAM_DIAGQUAD) {  // hdiag = w + Q' lambda : one pass over Q
    cols_dot(S, S.p_Q, S.ldj, S.m, S.n_loc, lam, 0);
    const double *cp = S.cpart, *w = S.p_w; double *hd = S.hdiag; int ns = S.m > 0 ? S.nsplit : 0; int64_t n = S.n_loc;
    const lfpsqp::IneqDev I = S.I; const bool ineq = S.ineq;
    // with bounds the augmented terms of inequality_helper.jl:144-158 are diagonal too: fold them into hdiag (2n entries)
    vec(S, n, [=] __device__(int64_t j, double *) {
      double s = split_sum(cp, ns, n, j, w[j]);
      if (ineq) { const double ly2 = 2.0 * I.lamy[j]; s += ly2 * I.q[j]; hd[n + j] = ly2 * I.s[j]; }
      hd[j] = s;
    });
    S.launches++;
  } else if (S.family == LFPSQP_FAM_SPARSE_QCQP) {  // values of H = P + sum_i lam_i Qc_i on the union pattern (fixed source order)
    const lfpsqp::SpqDev &D = S.spq;
    if (D.nh <= 0) return;
    const int grid = (int)std::min<int64_t>((D.nh + 255) / 256, 8 * (int64_t)S.sm_count);
    spq_hess_assemble_kernel<<<grid, 256, 0, S.stream>>>(D.nh, D.hsrc_ptr, D.hsrc_con, D.hsrc_val, lam, D.hval);
    S.launches++;
  }
}
// dest = H src, partial src.dest -> loop-partial slot 0 ; returns the number of partials written
static int fam_hess(LargeState &S, double *dest, const double *src, const double *x, const double *lam, int pred) {
  if (S.family == LFPSQP_FAM_HOST) {  // the caller has checked ctrl->status on the host (chunk = 1)
    cudaMemcpyAsync(S.hw, src, S.n_loc * sizeof(double), cudaMemcpyDeviceToHost, S.stream);
    cudaStreamSynchronize(S.stream);
    if (S.cb.hess_lag_vec(S.cb.user, S.hv, S.hw, S.hx, S.hlam, S.n, S.m)) S.cb_err = 1;
    cudaMemcpyAsync(dest, S.hv, S.n_loc * sizeof(double), cudaMemcpyHostToDevice, S.stream);
    if (!S.ineq) dot_partials_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.n_loc, src, dest, S.lp, 0, S.ctrl, pred);
    S.launches++;
    return S.vgrid;
  } else if (S.family == LFPSQP_FAM_DIAGQUAD) {
    const double *hd = S.hdiag; const LargeCtrl *ctrl = S.ctrl; double *lp = S.lp;
    // predicated elementwise kernel with the d.Ad partial (hdiag carries the bound terms: nv entries)
    hess_diag_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.nv, hd, src, dest, lp, ctrl, pred);
    S.launches++;
    return S.vgrid;
  } else if (S.family == LFPSQP_FAM_SPARSE_QCQP) {   // CSR pass over the assembled H; with bounds ineq_hess_aug_kernel writes the partial
    spq_csr(S, 2, S.spq.hrow, S.spq.hcol, S.spq.hval, S.spq.gh, src, dest, S.ineq ? nullptr : S.lp, pred);
    S.launches++;
    return S.vgrid;
  } else {
    const int np = (int)(S.n / 3), npl = (int)(S.n_loc / 3), i0 = (int)(S.col0 / 3);
    const double *xf = (S.world > 1) ? S.xfull_h : x;            // gathered by fam_hess_prepare
    const double *vf = thomson_gather(S, src, S.vfull);
    dim3 grid; thomson_grid(S, npl, grid);
    thomson_pair_kernel<2><<<grid, 256, 0, S.stream>>>(np, i0, npl, xf, vf, S.pairws, nullptr, 0, S.ctrl, pred);
    thomson_reduce_kernel<2><<<(3 * npl + 255) / 256, 256, 0, S.stream>>>(npl, grid.y, S.pairws, src, lam + i0, dest, S.lp, 0, S.ctrl, pred);
    S.launches += 2;
    return (3 * npl + 255) / 256;
  }
}

// Lagrangian Hessian action on the working vector: the family's on the x-half plus, with bounds, the augmented terms
// (augmented_hess_lag_vec!, inequality_helper.jl:144-158); src.dest partials -> loop slot 0
static int hess_apply(LargeState &S, double *dest, const double *src, int pred) {
  int nph = fam_hess(S, dest, src, S.x, S.lam, pred);
  if (S.ineq && S.family != LFPSQP_FAM_DIAGQUAD) {
    ineq_hess_aug_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.I, dest, src, S.lp, S.ctrl, pred);
    S.launches++;
    nph = S.vgrid;
  }
  return nph;
}

// ------------------------------------------------------------------ bound embedding: one-off elementwise operations
static void ineq_gradient(LargeState &S, const double *v) {  // inequality_gradient! (inequality_helper.jl:125-141)
  const lfpsqp::IneqDev I = S.I;
  vec(S, I.nx, [=] __device__(int64_t j, double *) {
    double Dx, Dy, Sv;
    ineq_grad(I.q[j], I.r[j], I.s[j], v[j], v[I.nx + j], Dx, Dy, Sv);
    I.Dx[j] = Dx; I.Dy[j] = Dy; I.S[j] = Sv;
  });
  S.launches++;
}
static void y_retract(LargeState &S, double *vn, const double *vb) {  // y_retract! (retractions.jl:451-500)
  const lfpsqp::IneqDev I = S.I;
  vec(S, I.nx, [=] __device__(int64_t j, double *) {
    double xn = vn[j], yn = vn[I.nx + j];
    ineq_yretract(I.q[j], I.r[j], I.s[j], I.t[j], vb[j], vb[I.nx + j], xn, yn);
    vn[j] = xn; vn[I.nx + j] = yn;
  });
  S.launches++;
}

template <class T> static bool dalloc(LargeState &S, T **p, size_t count);
// G (lower tiles) = Jg Jg'.  Jg is stored dense; unless it was found dense before, a one-pass scan marks the all-zero
// (64 rows x 16 columns) slabs and the SYRK skips K chunks that contribute nothing (Thomson: 24 of 768 chunks per diagonal tile).
static void gram_syrk(LargeState &S, const double *Jg) {
  const int m = S.m;
  GemmExt X; const GemmExt *ext = nullptr;
  if (S.gram_skip && S.gram_mode != 2 && S.nzmap && m > 64) {
    cudaMemsetAsync(&S.ctrl->nz_count, 0, sizeof(unsigned long long), S.stream);
    dim3 sg((unsigned)((S.n_loc + 1023) / 1024), (unsigned)S.nz_rows);
    zero_slab_map_kernel<<<sg, 256, 0, S.stream>>>(Jg, S.ldj, m, S.n_loc, S.nzmap, S.nz_ld, &S.ctrl->nz_count);
    S.launches++;
    X.nz = S.nzmap; X.nz_ld = S.nz_ld; X.nz_rows = S.nz_rows; ext = &X;
    if (S.gram_mode == 0) S.nz_pending = true;
    S.jmap_valid = (Jg == S.J);   // with bounds the map describes J diag(Dy), whose zeros are not J's
  } else S.jmap_valid = false;
  S.disp_syrk = true;
  gemm_nt(S, m, m, (int)S.n_loc, Jg, S.ldj, Jg, S.ldj, S.G, S.ldm, GEMM_ASSIGN, 1, ext);
  S.disp_syrk = false;
}
// S.G (lower triangle) = J J', or with bounds J diag(Dy^2) J' = PJct' PJct (optimize.jl:288-289 / SURVEY App. B), summed over
// the ranks.  timed: ev_g0 / ev_g1 bracket the product (the gram_ms of lfpsqp_large_factor).
static void gram(LargeState &S, bool timed) {
  const int m = S.m;
  const double *Jg = S.J;
  if (S.ineq && !S.csr) {   // SYRK operand Jw = J diag(Dy); the CSR Gram applies the weights itself
    dim3 sg((unsigned)std::min<int64_t>(std::max<int64_t>(((S.n_loc >> 1) + 255) / 256, 1), 32), (unsigned)std::min(m, 65535));
    ineq_scale_cols_kernel<<<sg, 256, 0, S.stream>>>(S.J, S.ldj, m, S.n_loc, S.I.Dy, S.Jw);
    S.launches++;
    Jg = S.Jw;
  }
  if (timed) cudaEventRecord(S.ev_g0, S.stream);
  if (S.csr) spj_gram(S);
  else gram_syrk(S, Jg);
  if (timed) cudaEventRecord(S.ev_g1, S.stream);
  if (S.world > 1) comm_allreduce(S, S.G, (size_t)m * S.ldm);
}
// Truncated path of optimize.jl:297-302 in Gram form: G = V diag(lambda) V' (Jacobi, large_eig.cu), G^+ into S.Ginv.
// regram: S.G no longer holds the Gram (a Cholesky attempt overwrote it) -> recompute it first.
static int factorize_pinv(lfpsqp_ctx *c, LargeState &S, bool regram) {
  const int m = S.m; const int64_t ldm = S.ldm;
  if (!S.eigV) {
    bool ok = dalloc(S, &S.eigV, (size_t)m * ldm) && dalloc(S, &S.eigT, (size_t)m * ldm) && dalloc(S, &S.eigLam, (size_t)m + 2) &&
              dalloc(S, &S.eigScratch, 40);
    if (ok && !S.Ginv) ok = dalloc(S, &S.Ginv, (size_t)m * ldm);
    if (!ok) return c->fail(LFPSQP_ERR_NOMEM, "rank-deficient path: workspace allocation failed");
  }
  if (regram) gram(S, false);
  unsigned long long *sc = S.eigScratch;
  if (large_eig_pinv_factors(S, S.G, S.eigV, S.eigLam, 1, reinterpret_cast<int *>(sc + 34), sc, reinterpret_cast<unsigned *>(sc + 32)))
    return c->fail(LFPSQP_ERR_CUDA, "rank-deficient path: cooperative launch of the Jacobi eigen-solver failed");
  dim3 tg((m + 31) / 32, (m + 31) / 32);
  transpose_kernel<<<tg, 256, 0, S.stream>>>(S.eigV, ldm, S.eigT, ldm, m, m);
  gemm_nt(S, m, m, m, S.eigT, ldm, S.eigT, ldm, S.Ginv, ldm, GEMM_ASSIGN, 0);   // G^+ = Vs' Vs
  S.pinv_active = true; S.prefer_pinv = true; S.explicit_inverse_ok = true; S.guard_pending = false;
  S.launches += 2; S.factorizations++;
  return 0;
}

// ------------------------------------------------------------------ factorisation of the Gram in S.G: G = L L', XT = L^-T, Linv = L^-1
static int factorize(lfpsqp_ctx *c, LargeState &S) {
  const int m = S.m; const int64_t ldm = S.ldm;
  S.invflag_valid = false;
  if (S.prefer_pinv) return factorize_pinv(c, S, false);   // this problem lost rank before: go straight to the eigen-decomposition
  S.pinv_active = false; S.rank_cur = m;
  diag_thresh_kernel<<<1, 256, 0, S.stream>>>(S.G, ldm, m, S.prm.eps_rank, S.thresh);
  constexpr int NB = 64;
  const size_t psm = 2 * NB * (NB + 1) * sizeof(double);
  int nblk = (m + NB - 1) / NB;
  // Block structure of G (and, with fill-in, of L): panel / trailing / inverse GEMM tiles whose operands are structurally zero
  // return at once.  A dense G costs one 15 us scan; a block-sparse one (Thomson: G is diagonal) keeps only the potf2 chain.
  GemmExt F1, F2, F3;
  const GemmExt *f1 = nullptr, *f2 = nullptr;
  int *done = nullptr;
  bool chain = true;
  if (S.blkflag && nblk > 1 && S.gram_skip) {
    block_nz_kernel<<<dim3(nblk, nblk), 256, 0, S.stream>>>(S.G, ldm, m, S.blkflag, nblk);
    S.launches++;
    F1.bf = S.blkflag; F1.bf_ld = nblk; F1.bf_n = nblk; F1.bf_mode = 1;
    F2 = F1; F2.bf_mode = 2; F3 = F1; F3.bf_mode = 3;
    f1 = &F1; f2 = &F2;
    done = S.blkflag + (size_t)nblk * nblk;
    // diagonal blocks nothing will ever update: factorised now, in parallel; the chain below skips them
    cudaMemsetAsync(&S.ctrl->g_dependent, 0, sizeof(int), S.stream);
    potf2_inv_indep_kernel<NB><<<nblk, 256, psm, S.stream>>>(S.G, ldm, m, S.Dblk, S.thresh, &S.ctrl->rankflag, S.blkflag, nblk, done,
                                                             &S.ctrl->g_dependent);
    S.launches++;
    if (S.g_blockdiag == 1) {   // block diagonal last time: look now (one short sync instead of ~5 launches per block)
      cudaMemcpyAsync(&S.hctrl->g_dependent, &S.ctrl->g_dependent, sizeof(int), cudaMemcpyDeviceToHost, S.stream);
      if (cudaStreamSynchronize(S.stream) == cudaSuccess && S.hctrl->g_dependent == 0) chain = false;
      else S.g_blockdiag = 0;
    } else S.gdep_pending = true;
  }
  // Right-looking blocked Cholesky with LOOK-AHEAD: the single-CTA factorisation of diagonal block b+1 (latency-bound, ~50 us)
  // runs on a second stream while the main stream applies the rank-NB update of block b to the rest of the trailing matrix.
  // Per block: potf2(b) -> L21 = A21 D' -> [panel part of the update: the nb2 columns of block b+1] -> event -> potf2(b+1) on
  // the side stream || [remaining trailing update] on the main stream.
  if (!S.side_stream) {
    cudaStreamCreateWithFlags(&S.side_stream, cudaStreamNonBlocking);
    cudaEventCreateWithFlags(&S.ev_panel, cudaEventDisableTiming); cudaEventCreateWithFlags(&S.ev_potf, cudaEventDisableTiming);
  }
  cudaStream_t main_s = S.stream, side_s = S.side_stream ? S.side_stream : S.stream;
  if (chain) { potf2_inv_kernel<NB><<<1, 256, psm, main_s>>>(S.G, ldm, std::min(NB, m), S.Dblk, S.thresh, &S.ctrl->rankflag, done, 0); S.launches++; }
  for (int b = 0; chain && b < nblk; b++) {
    int j0 = b * NB, nb = std::min(NB, m - j0), rem = m - j0 - nb;
    double *Db = S.Dblk + (size_t)b * NB * NB;
    if (rem <= 0) break;
    double *A21 = S.G + (int64_t)(j0 + nb) * ldm + j0;
    double *A22 = S.G + (int64_t)(j0 + nb) * ldm + (j0 + nb);
    F1.bf_a0 = b + 1; F1.bf_col = b;
    gemm_nt(S, rem, nb, nb, A21, ldm, Db, NB, A21, ldm, GEMM_ASSIGN, 0, f1);                     // L21 = A21 D'
    const int nb2 = std::min(NB, rem), rem2 = rem - nb2;
    F2.bf_a0 = b + 1; F2.bf_b0 = b + 1; F2.bf_col = b;
    gemm_nt(S, rem, nb2, nb, A21, ldm, A21, ldm, A22, ldm, GEMM_SUB, 0, f2);                     // panel of block b+1: A22[:, 0:nb2] -= L21 L21[0:nb2]'
    if (side_s != main_s) { cudaEventRecord(S.ev_panel, main_s); cudaStreamWaitEvent(side_s, S.ev_panel, 0); }
    potf2_inv_kernel<NB><<<1, 256, psm, side_s>>>(A22, ldm, nb2, S.Dblk + (size_t)(b + 1) * NB * NB, S.thresh, &S.ctrl->rankflag, done, b + 1);
    S.launches++;
    if (side_s != main_s) cudaEventRecord(S.ev_potf, side_s);
    if (rem2 > 0) {                                                                              // the rest of A22 -= L21 L21' (lower)
      F2.bf_a0 = b + 2; F2.bf_b0 = b + 2;
      gemm_nt(S, rem2, rem2, nb, A21 + (int64_t)nb2 * ldm, ldm, A21 + (int64_t)nb2 * ldm, ldm, A22 + (int64_t)nb2 * ldm + nb2, ldm, GEMM_SUB, 1, f2);
    }
    if (side_s != main_s) cudaStreamWaitEvent(main_s, S.ev_potf, 0);
  }
  // XT = L^-T (upper triangular, row-major) and Linv = L^-1 by recursive doubling from the inverted diagonal blocks:
  //   [L11 0; L21 L22]^-1 = [L11^-1 0; -L22^-1 L21 L11^-1, L22^-1]   i.e.  XT12 = -(XT11 L21') Linv22'
  // Per level (block size B = NB, 2 NB, ...): two batched DMMA GEMMs over all pairs of adjacent blocks (the triangular operand
  // bounds the K loop of each tile) + one batched transpose XT12 -> Linv21: 3 launches per level instead of 3 per block row.
  cudaMemsetAsync(S.XT, 0, (size_t)m * ldm * sizeof(double), S.stream);
  cudaMemsetAsync(S.Linv, 0, (size_t)m * ldm * sizeof(double), S.stream);
  diag_blocks_kernel<<<nblk, 256, 0, S.stream>>>(S.Dblk, NB, m, S.XT, S.Linv, ldm);
  S.launches++;
  for (int B = NB; chain && B < m; B *= 2) {   // (a block-diagonal L has a block-diagonal inverse: level 0 is all of it)
    const int nfull = m / (2 * B);                      // pairs with two complete blocks
    const int o_r = nfull * 2 * B, B2r = m - o_r - B;   // ragged last pair: L22 is B2r x B2r (if > 0)
    for (int part = 0; part < 2; part++) {
      const int np = part == 0 ? nfull : (B2r > 0 ? 1 : 0);
      if (np <= 0) continue;
      const int o = part == 0 ? 0 : o_r, B2 = part == 0 ? B : B2r;
      const int64_t pstride = (int64_t)2 * B * ldm + 2 * B;
      double *Tt = S.gemm_ws;                             // B x B2 per pair; row pitch B + 8: a power-of-two pitch made the
      const int64_t ldt = B + 8;                          // 128 rows of a tile hit the same L2 slices (second GEMM 1.5x slower)
      GemmExt e1 = f1 ? F3 : GemmExt();                    // a pair whose L21 is structurally zero keeps XT12 = 0 (memset above)
      if (f1) { e1.bf_r0 = (o + B) / NB; e1.bf_r1 = (o + B + B2 + NB - 1) / NB; e1.bf_c0 = o / NB; e1.bf_c1 = (o + B) / NB; e1.bf_batch = 2 * B / NB; }
      GemmExt e2 = e1;
      e1.batch = np; e1.batch_a = pstride; e1.batch_b = pstride; e1.batch_c = (int64_t)B * ldt; e1.tri = 1;
      gemm_nt(S, B, B2, B, S.XT + (int64_t)o * ldm + o, ldm, S.G + (int64_t)(o + B) * ldm + o, ldm, Tt, ldt, GEMM_ASSIGN, 0, &e1);
      e2.batch = np; e2.batch_a = (int64_t)B * ldt; e2.batch_b = pstride; e2.batch_c = pstride; e2.tri = 2;
      gemm_nt(S, B, B2, B2, Tt, ldt, S.Linv + (int64_t)(o + B) * ldm + (o + B), ldm, S.XT + (int64_t)o * ldm + (o + B), ldm, GEMM_ASSIGN_NEG, 0, &e2);
      dim3 tg((B2 + 31) / 32, (B + 31) / 32, np);
      transpose_kernel<<<tg, 256, 0, S.stream>>>(S.XT + (int64_t)o * ldm + (o + B), ldm, S.Linv + (int64_t)(o + B) * ldm + o, ldm, B, B2, pstride, pstride);
      S.launches++;
    }
  }
  // block structure of L^-1 for the unfused triangular passes (only worth it when G had structure: block-sparse J)
  S.invflag_valid = false;
  if (f1 && S.invflag && nblk <= 64 && S.gram_mode == 1) {
    block_nz_kernel<<<dim3(nblk, nblk), 256, 0, S.stream>>>(S.Linv, ldm, m, S.invflag, nblk);
    S.launches++;
    S.invflag_valid = true;
  }
  if (S.fused_ok && S.Ginv) {   // G^-1 = L^-T L^-1 = XT XT' for the fused projcg kernel (large_fused.cu): one more DMMA GEMM, m^3 flops
    gemm_nt(S, m, m, m, S.XT, ldm, S.XT, ldm, S.Ginv, ldm, GEMM_ASSIGN, 0);
    // guard of that shortcut: kappa = trace(G) * lambda_max(G^-1) >= cond(G) (8 power iterations on G^-1, ~0.1 ms); read_ctrl
    // turns it into S.explicit_inverse_ok
    const int nb = std::min(m, 64);
    lower_fro2_kernel<<<nb, 256, 0, S.stream>>>(S.G, ldm, m, S.gpart + 7 * (size_t)MAXP);
    power_step_kernel<<<1, 256, 0, S.stream>>>(m, nullptr, S.nr_t1, S.gpart + 7 * (size_t)MAXP, nb, S.ctrl);
    for (int it = 0; it < 8; it++) {
      rows_dot(S, S.Ginv, ldm, m, m, S.nr_t1, S.nr_t2, 0);
      power_step_kernel<<<1, 256, 0, S.stream>>>(m, S.nr_t2, S.nr_t1, nullptr, 0, S.ctrl);
    }
    S.launches += 10;
    S.guard_pending = true;
  }
  S.launches += 3;
  S.factorizations++;
  (void)c;
  return 0;
}

// v <- v - J'(J J')^-1 J v ; with lam_out the multipliers u = (J J')^-1 J v  (optimize.jl:306-307, :333-343 ; App. B)
// partial sums of the projected vector: slot0 = sum v^2, slot3 = max |v| (when want_norms)
// the passes over J of one projection: cpart = J' G^-1 J o with o = v, or with bounds o = Dy (Dy v_x - Dx v_y) (PJct' v);
// lam_out = G^-1 J o.  The elementwise tail (v - ...) is fused into the caller's next kernel.
static void proj_passes(LargeState &S, const double *v, double *lam_out, int pred) {
  const double *operand = v;
  if (S.ineq) {
    ineq_proj_pre_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.I, v, S.pb, S.ctrl, pred);
    S.launches++;
    operand = S.pb;
  }
  if (S.m <= 0) return;
  jrows(S, operand, S.tm, pred);
  if (S.world > 1) comm_allreduce(S, S.tm, S.m);
  gram_solve(S, S.tm, S.tu, lam_out, pred);
  jcols(S, S.tu, pred);
}
static void project(LargeState &S, double *v, double *lam_out, int pred, int want_norms, int want_mult = 0) {
  proj_passes(S, v, lam_out, pred);
  const double *cp = S.cpart; int ns = S.m > 0 ? S.jsplit : 0; int64_t n = S.n_loc;
  if (!S.ineq) {
    vec(S, n, [=] __device__(int64_t j, double *acc) {
      const double s = split_sum(cp, ns, n, j);
      double r = v[j] - s; v[j] = r;
      acc[0] += r * r; acc[3] = nanmax(acc[3], fabs(r));
    }, 0, want_norms ? 1 : 0, want_norms);
  } else {  // d - Q Q'd (optimize.jl:314-317) and lambda_y (calculate_lambda_kkt!, inequality_helper.jl:286-308)
    const lfpsqp::IneqDev I = S.I;
    vec(S, n, [=] __device__(int64_t j, double *acc) {
      double ox, oy, aa, wj;
      ineq_proj_tail(I, j, v[j], v[I.nx + j], cp, ns, ox, oy, aa, wj);
      v[j] = ox; v[I.nx + j] = oy;
      if (want_mult) I.lamy[j] = -1.0 * (I.Dx[j] / I.S[j]) * wj + aa / I.S[j];
      acc[0] += ox * ox + oy * oy; acc[3] = nanmax(acc[3], nanmax(fabs(ox), fabs(oy)));
    }, 0, want_norms ? 1 : 0, want_norms);
  }
  S.launches++;
}

// ------------------------------------------------------------------ projcg! (projcg.jl:40-121), c = 0
// b = S.d (projected -grad). Solution -> S.nd. Fills S.hctrl (status/iter/nr) on return.
// cvec (device, m doubles, replicated) selects the general form of projcg.jl:55: x0 = U c, r = A x0 - b, with U the
// Cholesky-QR basis J' L^-T (orthonormal columns spanning the same space as the reference's U; SURVEY App. B); the
// driver always passes c = 0 (cvec = nullptr).  lam_out receives U'(b - A x) (projcg.jl:115-118).
static int projcg(lfpsqp_ctx *c, LargeState &S, double tol, int64_t maxit, int chunk, const double *cvec = nullptr,
                  double *lam_out = nullptr) {
  const int64_t n = S.nv;   // working length: n_loc, or 2 n_loc with bounds
  const int ns = S.m > 0 ? S.jsplit : 0;
  double *xs = S.nd, *r = S.w0, *dc = S.w1, *Ad = S.w2, *rp = S.w3, *gp = S.w4;
  const double *b = S.d;
  if (S.family == LFPSQP_FAM_HOST) chunk = 1;   // the Hessian callback runs on the host: one status check per iteration
  if (cvec && S.m > 0 && !S.ineq) {
    tri_gemv(S, 1, cvec, S.tu, nullptr, 0);   // L^-T c
    jcols(S, S.tu, 0);
    const double *cp = S.cpart; const int64_t nl = S.n_loc;
    vec(S, n, [=] __device__(int64_t j, double *) { xs[j] = split_sum(cp, ns, nl, j); });
    hess_apply(S, r, xs, 0);
    vec(S, n, [=] __device__(int64_t i, double *) { r[i] -= b[i]; });
    S.launches += 2;
  } else
  vec(S, n, [=] __device__(int64_t i, double *) { xs[i] = 0.0; r[i] = -b[i]; });
  // g = r - U U' r (projcg.jl:59-60) ; r = g ; d = -g ; rg partials -> loop slot 3 (= 2 + (par^1) for k = 0)
  proj_passes(S, r, nullptr, 0);
  if (S.ineq) ineq_cg_init_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.I, r, dc, S.cpart, ns, S.lp);
  else cg_init_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, r, dc, S.cpart, ns, S.lp);
  if (S.world > 1) comm_allreduce_loop_slot(S, 3, S.np_loop_raw);
  S.launches += 2;
  // min(maxit, n + length(c)) (projcg.jl:71): c has length rank = m, or n + rank with the bound projector (optimize.jl:366-372)
  const int64_t rk = S.pinv_active ? S.rank_cur : S.m;
  int64_t lim = std::min<int64_t>(maxit, S.ineq ? 3 * S.n + rk : S.n + rk);
  S.hctrl->tol = tol; S.hctrl->lim = (int)std::min<int64_t>(lim, 2000000000); S.hctrl->iter = 0; S.hctrl->status = (lim > 0) ? 0 : 4;
  S.hctrl->nr = INFINITY;
  write_ctrl_fields(S);
  int64_t k = 0;
  // persistent fused path (large_fused.cu): one cooperative kernel per chunk instead of 8 launches per iteration
  bool fused = S.fused_ok && lim > 0 && !cvec;
  while (fused && S.hctrl->status == 0) {
    if (fused_projcg_chunk(S, std::max(4 * chunk, 64), k == 0, xs, r, dc, Ad, rp, gp)) {
      if (k == 0) { fused = false; break; }          // not eligible / launch refused before anything ran: unfused path
      return -1;
    }
    k++;
    if (read_ctrl(c, S)) return -1;
  }
  while (!fused && S.hctrl->status == 0) {
    for (int q = 0; q < chunk; q++, k++) {
      const int par = (int)(k & 1);
      int nph = hess_apply(S, Ad, dc, 1);
      if (S.world > 1) comm_allreduce_loop_slot(S, 0, nph), nph = 1;
      cg_update1_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, xs, dc, r, Ad, rp, S.lp, nph, S.np_loop, par, S.ctrl);
      proj_passes(S, rp, nullptr, 1);
      if (S.ineq) ineq_cg_update2_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.I, rp, gp, S.cpart, ns, S.lp, par, S.ctrl, 1);
      else cg_update2_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, rp, gp, S.cpart, ns, S.lp, par, S.ctrl, 1);
      if (S.world > 1) comm_allreduce_loop_slots_cg(S, par);
      cg_update3_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, dc, r, gp, S.lp, S.np_loop, par, S.ctrl);
      S.launches += 3;
    }
    if (read_ctrl(c, S) || S.cb_err) return -1;
  }
  S.projcg_iters += S.hctrl->iter;
  if (S.hctrl->status == 2) {  // negative curvature: x = d/|d| (projcg.jl:77-82)
    S.projcg_negcurv++;
    vec(S, n, [=] __device__(int64_t i, double *acc) { acc[0] += dc[i] * dc[i]; }, 0, 1);
    finalize(S, 1u, 0);
    const LargeCtrl *ctrl = S.ctrl;
    vec(S, n, [=] __device__(int64_t i, double *) { xs[i] = dc[i] / sqrt(ctrl->s[0]); });
    S.launches += 2;
    S.hctrl->nr = INFINITY;
  }
  if (lam_out && S.m > 0 && !S.ineq) {   // lambda = U'(b - A x) (projcg.jl:115-118) = L^-1 J (b - A x); NaN after a negative-curvature exit (:80)
    if (S.hctrl->status == 2) {
      vec(S, S.m, [=] __device__(int64_t a, double *) { lam_out[a] = NAN; });
    } else {
      const int st_keep = S.hctrl->status;
      hess_apply(S, Ad, xs, 0);
      vec(S, n, [=] __device__(int64_t i, double *) { Ad[i] = b[i] - Ad[i]; });
      jrows(S, Ad, S.tm, 0);
      if (S.world > 1) comm_allreduce(S, S.tm, S.m);
      tri_gemv(S, 0, S.tm, lam_out, nullptr, 0);
      S.launches++;
      (void)st_keep;
    }
  }
  return 0;
}

// ------------------------------------------------------------------ pcg! (retractions.jl:179-246), M! = copy, on (J'J + mu I) dx = r
// state: dx = S.w3 (initial guess), r = S.w0 (= b - A dx), p = S.w1 (zeroed by the caller), z = S.w2;
// r.r partials of the start residual in loop slot 5.  Device-predicated, enqueued in chunks.
static int run_pcg(lfpsqp_ctx *c, LargeState &S, double mu, double tol, int64_t maxiter) {
  const int64_t n = S.nv, nx = S.n_loc; const int m = S.m;
  double *r = S.w0, *pv = S.w1, *z = S.w2, *dx = S.w3;
  S.hctrl->tol = tol; S.hctrl->mu = mu; S.hctrl->pcg_iter = 0; S.hctrl->pcg_lim = (int)std::min<int64_t>(maxiter, 2000000000); S.hctrl->pcg_status = 0;
  write_ctrl_fields(S);
  int64_t k = 0;
  // persistent fused path (large_fused.cu): the whole pcg! call is one cooperative launch
  if (S.fused_ok && maxiter <= 128 && fused_pcg(S, dx, r, pv, z) == 0) return read_ctrl(c, S) ? -1 : 0;
  while (S.hctrl->pcg_status == 0) {
    for (int q = 0; q < S.pcg_chunk; q++, k++) {
      const int par = (int)(k & 1);
      if (S.world > 1) comm_allreduce_loop_slot(S, 5 + par, S.np_loop_raw);
      pcg_a_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, pv, r, S.lp, S.np_loop, par, k == 0, S.ctrl);
      jrows(S, pv, S.tm, 2);                          // J p_x (bigA' p = [S (Dx p_x + Dy p_y) ; J p_x] with bounds)
      if (S.world > 1) comm_allreduce(S, S.tm, m);
      jcols(S, S.tm, 2);
      if (S.ineq) ineq_pcg_z_kernel<<<S.vgrid, 256, 0, S.stream>>>(S.I, z, pv, S.cpart, S.jsplit, S.lp, S.ctrl);
      else pcg_z_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, z, pv, S.cpart, S.jsplit, S.lp, S.ctrl);
      if (S.world > 1) comm_allreduce_loop_slot(S, 4, S.np_loop_raw);
      pcg_x_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, dx, r, pv, z, S.lp, S.np_loop, par, S.ctrl);
      S.launches += 3;
    }
    if (read_ctrl(c, S)) return -1;
  }
  return 0;
}

// ------------------------------------------------------------------ retract!(::ProjPenalty) (retractions.jl:265-441) + pcg! (:179-246)
// xtil -> xnew ; returns flag, it1 (outer), it2 (pcg total)
static int retract_pp(lfpsqp_ctx *c, LargeState &S, int *flag_out, int *it1, int *it2) {
  const int64_t n = S.n_loc, nv = S.nv; const int m = S.m;
  const bool ineq = S.ineq; const lfpsqp::IneqDev I = S.I;
  double *r = S.w0, *pv = S.w1, *z = S.w2, *dx = S.w3, *gv = S.w4, *xnew = S.xnew, *cval = S.cval, *cvh = S.cvh, *cvc = S.cvc;
  const double *xtil = S.xtil;
  const lfpsqp_params &prm = S.prm;
  auto hmax = [](double a, double b) { return (b > a || std::isnan(b)) ? b : a; };
  int flag = 0;
  (void)z;
  cudaMemcpyAsync(xnew, xtil, nv * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);
  double mu = prm.mu0;
  int i = 0, pcg_total = 0;
  while (i < prm.maxiter_retract) {
    fam_c_jac(S, true, cval, xnew);                                                       // :340
    // curtol = |c|_inf (slot 3 max), c.c (slot 0) ; with bounds also |h|_inf (slot 4), h.h (slot 1) and the stale tail
    if (!ineq) {
      vec(S, m, [=] __device__(int64_t a, double *acc) { double v = cval[a]; acc[0] += v * v; acc[3] = nanmax(acc[3], fabs(v)); }, 0, 1, 1);
    } else {
      // inequality_gradient! on the shared decomposition (:343-347) ; h -> cvalaug[1:n] (:350)
      vec(S, n, [=] __device__(int64_t j, double *acc) {
        const double xv = xnew[j], yv = xnew[n + j];
        double Dx, Dy, Sv;
        ineq_grad(I.q[j], I.r[j], I.s[j], xv, yv, Dx, Dy, Sv);
        I.Dx[j] = Dx; I.Dy[j] = Dy; I.S[j] = Sv;
        const double h = ineq_h(I.q[j], I.r[j], I.s[j], I.t[j], xv, yv);
        cvh[j] = h; acc[0] += h * h; acc[3] = nanmax(acc[3], fabs(h));
      }, 1, 1, 1);
      // :352 takes the norm of ALL of cvalaug, whose tail still holds the previous c values; then :356 refreshes the tail
      vec(S, m, [=] __device__(int64_t a, double *acc) {
        const double v = cval[a];
        acc[3] = nanmax(acc[3], nanmax(fabs(v), fabs(cvc[a])));
        cvc[a] = v; acc[0] += v * v;
      }, 0, 1, 1);
      S.launches++;
    }
    // g = xnew - xtilde, g.g (slot 2)
    vec(S, nv, [=] __device__(int64_t k, double *acc) { double t = xnew[k] - xtil[k]; gv[k] = t; acc[0] += t * t; }, 2, 1);
    finalize(S, ineq ? (1u | 2u | 4u) : (1u | 4u), ineq ? (8u | 16u) : 8u, 1u | 8u);
    S.launches += 2;
    if (read_ctrl(c, S) || S.cb_err) return -1;
    const double curtol = ineq ? hmax(S.hctrl->s[3], S.hctrl->s[4]) : S.hctrl->s[3];
    const double cc = S.hctrl->s[0], hh = ineq ? S.hctrl->s[1] : 0.0, gg = S.hctrl->s[2];
    if (curtol < prm.eps_c) break;                                                       // :359-361
    const double prev_obj = (hh + cc) + mu * gg;                                         // :366
    // g = J' c + mu g, or bigA [h ; c] + mu g (:369) ; dx = 0 ; r = g ; r.r partials -> loop slot 5 (rho_0)
    jcols(S, cval, 0);
    if (ineq) ineq_pp_rhs_kernel<<<S.vgrid, 256, 0, S.stream>>>(I, gv, dx, r, pv, S.cpart, S.jsplit, mu, cvh, S.lp);
    else pp_rhs_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, gv, dx, r, pv, S.cpart, S.jsplit, mu, S.lp);
    S.launches++;
    if (run_pcg(c, S, mu, prm.eps_c, prm.maxiter_pcg)) return -1;                       // :375
    int pcg_i = S.hctrl->pcg_iter;
    pcg_total += pcg_i;
    if (pcg_i == prm.maxiter_pcg) { flag = 2; break; }                                   // :240-243, :377-381
    // inner Armijo (:384-426)
    vec(S, nv, [=] __device__(int64_t q, double *acc) {
      double xk = xnew[q]; pv[q] = xk;
      acc[0] += gv[q] * dx[q];                     // ar_dot = -g.dx
      xk -= dx[q]; xnew[q] = xk;
      double t = xk - xtil[q]; gv[q] = t; acc[1] += t * t;
    }, 0, 2);
    fam_c_jac(S, false, cval, xnew);                                                    // :392
    vec(S, m, [=] __device__(int64_t a, double *acc) { double v = cval[a]; if (ineq) cvc[a] = v; acc[0] += v * v; }, 2, 1);   // slot 2 only
    if (ineq) {                                                                           // h -> cvalaug[1:n] (:395-397), slot 4
      vec(S, n, [=] __device__(int64_t j, double *acc) {
        const double h = ineq_h(I.q[j], I.r[j], I.s[j], I.t[j], xnew[j], xnew[n + j]);
        cvh[j] = h; acc[0] += h * h;
      }, 4, 1);
      S.launches++;
    }
    S.launches += 2;
    finalize(S, ineq ? (7u | 16u) : 7u, 0, 4u);
    if (read_ctrl(c, S) || S.cb_err) return -1;
    double ar_dot = -S.hctrl->s[0], dist2 = S.hctrl->s[1], ccnew = S.hctrl->s[2], hhnew = ineq ? S.hctrl->s[4] : 0.0;
    double alpha = 1.0;
    int armijo_count = 0;
    while ((hhnew + ccnew) + mu * dist2 > prev_obj + 1e-4 * alpha * ar_dot) {            // :403
      alpha /= 2;
      double al = alpha;
      vec(S, nv, [=] __device__(int64_t q, double *acc) {
        double xk = pv[q] - al * dx[q]; xnew[q] = xk;
        double t = xk - xtil[q]; gv[q] = t; acc[0] += t * t;
      }, 1, 1);                                                                           // slot 1 only
      S.launches++;
      if (ineq) {   // :413-415: the bound part of the merit IS refreshed during backtracking
        vec(S, n, [=] __device__(int64_t j, double *acc) {
          const double h = ineq_h(I.q[j], I.r[j], I.s[j], I.t[j], xnew[j], xnew[n + j]);
          cvh[j] = h; acc[0] += h * h;
        }, 4, 1);
        S.launches++;
      }
      finalize(S, ineq ? (2u | 16u) : 2u, 0);
      if (read_ctrl(c, S)) return -1;
      dist2 = S.hctrl->s[1];
      if (ineq) hhnew = S.hctrl->s[4];
      // :410-417: the c-part of the merit stays frozen at its alpha = 1 value (stale cval quirk)
      armijo_count++; S.pp_backtracks++;
      if (armijo_count == 100) { flag = 3; break; }
    }
    i++;
    mu = std::min(mu * 0.1, sqrt(hhnew + ccnew));                                        // :431 (norm of the stale cvalaug)
  }
  if (i == prm.maxiter_retract) flag = 1;
  *flag_out = flag; *it1 = i; *it2 = pcg_total;
  return 0;
}

// ------------------------------------------------------------------ retract!(::NR) (retractions.jl:75-177), Cholesky-QR basis (App. B)
static int retract_nr(lfpsqp_ctx *c, LargeState &S, int *flag_out, int *it1) {
  const int64_t n = S.n_loc; const int m = S.m; const int64_t ldm = S.ldm;
  double *xnew = S.xnew, *cval = S.cval, *D = S.Dnr, *t1 = S.nr_t1, *t2 = S.nr_t2, *dcv = S.nr_dc;
  const bool ineq = S.ineq; const lfpsqp::IneqDev I = S.I; const double *xb = S.x;
  cudaMemcpyAsync(xnew, S.xtil, S.nv * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);
  if (ineq) y_retract(S, xnew, xb);                                                      // :118-123
  fam_c_jac(S, false, cval, xnew);
  cudaMemcpyAsync(D, S.Linv, (size_t)m * ldm * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);   // D0 = L^-1
  int i = 0;
  while (i < S.prm.maxiter_retract) {
    vec(S, m, [=] __device__(int64_t a, double *acc) { acc[3] = nanmax(acc[3], fabs(cval[a])); }, 0, 0, 1);
    finalize(S, 0, 8u, 8u);
    if (read_ctrl(c, S) || S.cb_err) return -1;
    if (S.hctrl->s[3] < S.prm.eps_c) break;                                              // :135
    rows_dot(S, D, ldm, m, m, cval, t1, 0);                                              // D c
    vec(S, m, [=] __device__(int64_t a, double *) { t1[a] = -t1[a]; });                   // :140 delta = -D c
    // xnew += Q delta, Q = J' L^-T (:141)
    tri_gemv(S, 1, t1, S.tu, nullptr, 0);
    jcols(S, S.tu, 0);
    { const double *cp = S.cpart; int ns = S.jsplit;
      // with bounds the basis is Q = PJct L^-T: x += Dy^2 w, y -= Dx Dy w, then y_retract! (:141-143)
      vec(S, n, [=] __device__(int64_t j, double *) {
        const double s = split_sum(cp, ns, n, j);
        if (!ineq) { xnew[j] += s; return; }
        const double dx = I.Dx[j], dy = I.Dy[j];
        double xn = xnew[j] + dy * dy * s, yn = xnew[n + j] - dx * dy * s;
        ineq_yretract(I.q[j], I.r[j], I.s[j], I.t[j], xb[j], xb[n + j], xn, yn);
        xnew[j] = xn; xnew[n + j] = yn;
      }); }
    fam_c_jac(S, false, t2, xnew);                                                     // :144-149
    vec(S, m, [=] __device__(int64_t a, double *) { dcv[a] = t2[a] - cval[a]; cval[a] = t2[a]; });
    // Good Broyden (:156-160): t2 = D' delta ; t1 = delta - D dc ; D += t1 t2' / (t2.dc)
    {
      dim3 grid((unsigned)((m + 511) / 512), S.nsplit);
      cols_dot_kernel<false><<<grid, 256, S.rows_per_split * sizeof(double), S.stream>>>(D, ldm, m, m, t1, S.cpart, S.rows_per_split, S.ctrl, 0);
      const double *cp = S.cpart; int ns = S.nsplit;
      vec(S, m, [=] __device__(int64_t a, double *acc) {
        const double s = split_sum(cp, ns, m, a);
        t2[a] = s; acc[0] += s * dcv[a];
      }, 0, 1);
      finalize(S, 1u, 0, 1u);
      rows_dot(S, D, ldm, m, m, dcv, S.tm, 0);
      double *tmv = S.tm;
      vec(S, m, [=] __device__(int64_t a, double *) { t1[a] -= tmv[a]; });
      const LargeCtrl *ctrl = S.ctrl;
      vec(S, (int64_t)m * m, [=] __device__(int64_t e, double *) {
        int rr = (int)(e / m), cc2 = (int)(e % m);
        D[(int64_t)rr * ldm + cc2] += (1.0 / ctrl->s[0]) * t1[rr] * t2[cc2];
      });
    }
    S.launches += 8;
    i++;
  }
  *flag_out = (i == S.prm.maxiter_retract) ? 1 : 0; *it1 = i;
  return 0;
}

// one trial point of a line search: xtil = x + al d, retracted into xnew by kind 0 Euclidean (a copy), 1 YRetract, 2 NR or
// 3 ProjPenalty; flag = the retraction's flag (0 for kinds 0 and 1)
static int retract_trial(lfpsqp_ctx *c, LargeState &S, int kind, double al, int *flag) {
  const double *x = S.x, *d = S.d; double *xtil = S.xtil;
  vec(S, S.nv, [=] __device__(int64_t i, double *) { xtil[i] = x[i] + al * d[i]; });
  int rc = 0, i1 = 0, i2 = 0;
  *flag = 0;
  if (kind <= 1) {
    cudaMemcpyAsync(S.xnew, xtil, S.nv * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);
    if (kind == 1) y_retract(S, S.xnew, x);
  } else if (kind == 2) rc = retract_nr(c, S, flag, &i1);
  else rc = retract_pp(c, S, flag, &i1, &i2);
  S.retract_outer += i1; S.retract_pcg += i2; S.armijo_trials++;
  return rc;
}

// ------------------------------------------------------------------ exact_linesearch! (linesearch.jl:107-339), host control flow
static int exact_linesearch(lfpsqp_ctx *c, LargeState &S, int kind, double fval, double *newf_o, double *f_diff_o,
                            double *step_diff_o, int *flag_o) {
  const int64_t n = S.nv;
  const lfpsqp_params &prm = S.prm;
  const double phi1 = (3.0 - sqrt(5.0)) / 2.0, phi2 = (sqrt(5.0) - 1.0) / 2.0, phi3 = (sqrt(5.0) + 1.0) / 2.0;
  double Delta = prm.alpha, f_a = 0, f_b = 0, f_c = 0, f_d = 0, a_a = 0, a_b = 0, a_c = 0, a_d = 0;
  double *x_a = S.ex[0], *x_b = S.ex[1], *x_c = S.ex[2], *x_d = S.ex[3], *swp;
  const double *x = S.x, *d = S.d; double *xnew = S.xnew;
  bool do_shrinking = true;
  int flag = 0, rc = 0;
  auto TRIAL = [&](double *pt, double al) {
    rc |= retract_trial(c, S, kind, al, &flag);
    cudaMemcpyAsync(pt, xnew, n * 8, cudaMemcpyDeviceToDevice, S.stream);
  };
  auto FVAL = [&](const double *pt) -> double {
    fam_f(S, pt); finalize(S, 1u, 0);
    if (read_ctrl(c, S) || S.cb_err) { rc = -1; return NAN; }
    return S.hctrl->s[0];
  };
  cudaMemcpyAsync(x_d, x, n * 8, cudaMemcpyDeviceToDevice, S.stream); f_d = fval;
  while (true) {
    swp = x_b; x_b = x_c; x_c = x_d; x_d = swp;
    f_b = f_c; f_c = f_d; a_b = a_c; a_c = a_d;
    TRIAL(x_d, a_d + Delta);
    a_d += Delta;
    if (rc) return -1;
    if (flag > 0 || a_d > 1.0) { f_d = INFINITY; break; }
    f_d = FVAL(x_d);
    if (f_d > f_c) break;
    do_shrinking = false;
    Delta *= phi3;
  }
  if (do_shrinking) {
    f_b = fval; a_b = 0.0; cudaMemcpyAsync(x_b, x, n * 8, cudaMemcpyDeviceToDevice, S.stream);
    f_c = INFINITY; a_c = Delta;
    swp = x_d; x_d = x_c; x_c = swp;
    while (true) {
      swp = x_d; x_d = x_c; x_c = swp;
      f_d = f_c; a_d = a_c;
      TRIAL(x_c, phi1 * a_c);
      a_c *= phi1;
      if (rc) return -1;
      if (flag > 0 || a_c > 1.0) f_c = INFINITY; else f_c = FVAL(x_c);
      if (f_c <= fval || a_c < 1e-100) break;
    }
  }
  f_a = f_b; f_b = f_c; a_a = a_b; a_b = a_c;
  swp = x_a; x_a = x_b; x_b = x_c; x_c = swp;
  a_c = a_a + phi2 * (a_d - a_a);
  TRIAL(x_c, a_c);
  if (rc) return -1;
  if (flag > 0 || a_c > 1.0) f_c = INFINITY; else f_c = FVAL(x_c);
  vec(S, n, [=] __device__(int64_t i, double *acc) { acc[0] += d[i] * d[i]; }, 0, 1);
  finalize(S, 1u, 0);
  if (read_ctrl(c, S)) return -1;
  const double nd_ = sqrt(S.hctrl->s[0]);
  while ((a_c - a_b) > 1e-6 * nd_) {
    if (f_b < f_c || isinf(f_c)) {
      swp = x_d; x_d = x_c; x_c = x_b; x_b = swp;
      f_d = f_c; f_c = f_b; a_d = a_c; a_c = a_b;
      a_b = a_a + phi1 * (a_d - a_a);
      TRIAL(x_b, a_b);
      f_b = FVAL(x_b);
    } else {
      swp = x_a; x_a = x_b; x_b = x_c; x_c = swp;
      f_a = f_b; f_b = f_c; a_a = a_b; a_b = a_c;
      a_c = a_a + phi2 * (a_d - a_a);
      TRIAL(x_c, a_c);
      if (flag > 0 || a_c > 1.0) f_c = INFINITY; else f_c = FVAL(x_c);
    }
    if (rc) return -1;
  }
  (void)f_a; (void)f_d;
  double newf;
  if (f_b < f_c) { cudaMemcpyAsync(xnew, x_b, n * 8, cudaMemcpyDeviceToDevice, S.stream); newf = f_b; }
  else { cudaMemcpyAsync(xnew, x_c, n * 8, cudaMemcpyDeviceToDevice, S.stream); newf = f_c; }
  vec(S, S.n_loc, [=] __device__(int64_t i, double *acc) { double t = xnew[i] - x[i]; acc[0] += t * t; }, 0, 1);   // first n entries
  finalize(S, 1u, 0);
  if (read_ctrl(c, S)) return -1;
  *step_diff_o = sqrt(S.hctrl->s[0]); *f_diff_o = fabs(newf - fval); *newf_o = newf; *flag_o = flag;
  return 0;
}

// ------------------------------------------------------------------ the driver (optimize.jl:119-443)
static int solve(lfpsqp_ctx *c, LargeState &S, const double *x0_host, double *x_out, double *obj_hist, int64_t H,
                 int64_t *obj_len, double *lambda, lfpsqp_term *term, lfpsqp_stats *stats) {
  const int64_t n = S.n_loc, nv = S.nv; const int m = S.m;
  const bool ineq = S.ineq; const lfpsqp::IneqDev I = S.I;
  const lfpsqp_params &prm = S.prm;
  double *x = S.x, *g = S.g, *d = S.d, *xnew = S.xnew, *xtil = S.xtil, *nd = S.nd;
  S.reset_counters();
  S.cb_err = 0;
  S.prefer_pinv = false; S.pinv_active = false; S.rank_cur = m;
  CK(cudaMemcpyAsync(x, x0_host, n * sizeof(double), cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemsetAsync(g, 0, nv * sizeof(double), S.stream));                              // g[n+1:] == 0 (optimize.jl:191)
  if (m > 0) CK(cudaMemsetAsync(S.cvc, 0, m * sizeof(double), S.stream));
  if (ineq) {                                                                            // x = [x0 ; y0] (optimize.jl:176-182)
    vec(S, n, [=] __device__(int64_t j, double *) { x[n + j] = ineq_y0(I.q[j], I.r[j], I.s[j], I.t[j], x[j]); });
    CK(cudaMemsetAsync(S.cvh, 0, n * sizeof(double), S.stream));
  }
  reset_ctrl(S);
  int64_t it = 0, nobj = 0;
  double f_diff = INFINITY, step_diff = INFINITY, kkt_diff = INFINITY, prev_grad_norm = 0.0;
  fam_f(S, x); finalize(S, 1u, 0);
  if (m > 0) fam_c_jac(S, false, S.cval, x);                                          // :252
  if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
  if (S.cb_err) return LFPSQP_ERR_CALLBACK;
  double fval = S.hctrl->s[0];
  if (nobj < H) obj_hist[nobj] = fval;
  nobj++;
  int cond = LFPSQP_F_TOL, status = 0, last_flag = 0;
  while (true) {
    fam_grad(S, g, x);                                                                  // :259
    vec(S, nv, [=] __device__(int64_t i, double *) { d[i] = -1.0 * g[i]; });             // :262
    S.launches++;
    if (prm.beta > 0 && S.cb.randn) {                                                   // :264-273, randn! from the caller's RNG
      if (S.cb.randn(S.cb.user, S.hw, nv)) S.cb_err = 1;
      double *noise = S.w0;
      CK(cudaMemcpyAsync(noise, S.hw, nv * sizeof(double), cudaMemcpyHostToDevice, S.stream));
      const double coef = prm.t_beta > 0 ? prm.beta * fmax(1.0 - (double)it / (double)prm.t_beta, 0.0) : prm.beta;
      vec(S, nv, [=] __device__(int64_t i, double *) { d[i] += coef * noise[i]; });
      CK(cudaStreamSynchronize(S.stream));   // S.hw is reused by the next callback
    } else if (prm.beta > 0 && it < S.noise_T) {                                        // device families: the caller's noise rows
      const double coef = prm.t_beta > 0 ? prm.beta * fmax(1.0 - (double)it / (double)prm.t_beta, 0.0) : prm.beta;
      const double *noise = S.noise_dev + (size_t)it * nv;
      vec(S, nv, [=] __device__(int64_t i, double *) { d[i] += coef * noise[i]; });
      S.launches++;
    }
    if (ineq) ineq_gradient(S, x);                                                      // :277
    if (m > 0 || ineq) {
      const double tf0 = now_ms();
      if (m > 0) {
        fam_c_jac(S, true, S.cval, x);                                                   // :283
        gram(S, true);
        if (factorize(c, S)) return LFPSQP_ERR_CUDA;
        cudaMemcpyAsync(xtil, d, nv * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);   // d before the projection (rank-loss redo)
      }
      project(S, d, S.lam, 0, 1, 1);                                                    // :306-307 / :314-317, :331-343
      S.t_factor_pending = tf0;
    } else {
      vec(S, n, [=] __device__(int64_t i, double *acc) { double r = d[i]; acc[0] += r * r; acc[3] = nanmax(acc[3], fabs(r)); }, 0, 1, 1);
    }
    finalize(S, 1u, 8u);
    if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
    if (S.cb_err) return LFPSQP_ERR_CALLBACK;
    if (S.t_factor_pending > 0) { S.ms_factor += now_ms() - S.t_factor_pending; S.t_factor_pending = 0; }
    if (S.hctrl->rankflag) {
      // the Cholesky pivot test failed: the reference's truncated path (optimize.jl:297-302, :335-340) through the
      // eigen-decomposition of the Gram; the projection is redone with the pseudo-inverse
      S.hctrl->rankflag = 0; write_ctrl_fields(S);
      if (factorize_pinv(c, S, true)) return LFPSQP_ERR_CUDA;
      cudaMemcpyAsync(d, xtil, nv * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);
      project(S, d, S.lam, 0, 1, 1);
      finalize(S, 1u, 8u);
      if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
    }
    if (S.pinv_active) { S.rank_cur = (int)S.hctrl->s[14]; status |= LFPSQP_ST_RANK_DEFICIENT; }   // informational, as in batched mode
    kkt_diff = S.hctrl->s[3];                                                           // :320
    double gn = sqrt(S.hctrl->s[0]);
    if (f_diff <= prm.eps_f) { cond = LFPSQP_F_TOL; break; }                            // :347-359
    else if (step_diff <= prm.eps_x) { cond = LFPSQP_X_TOL; break; }
    else if (it >= prm.maxiter) { cond = LFPSQP_MAX_ITER; break; }
    else if (kkt_diff <= prm.eps_kkt) { cond = LFPSQP_KKT_TOL; break; }
    if (!(kkt_diff == kkt_diff)) { status |= LFPSQP_ST_NONFINITE; cond = LFPSQP_MAX_ITER; break; }
    if (prm.do_newton) {                                                                // :364-390
      double tol = prm.tn_kappa * fmin(1.0, gn / prev_grad_norm) * gn;
      prev_grad_norm = gn;
      const double tp0 = now_ms();
      fam_hess_prepare(S, x, S.lam);
      if (projcg(c, S, tol, prm.tn_maxiter, S.cg_chunk)) return S.cb_err ? LFPSQP_ERR_CALLBACK : LFPSQP_ERR_CUDA;
      S.ms_projcg += now_ms() - tp0;
      vec(S, nv, [=] __device__(int64_t i, double *acc) { acc[0] += nd[i] * d[i]; }, 0, 1);
      finalize(S, 1u, 0);
      if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
      if (S.hctrl->s[0] > 0.0) { cudaMemcpyAsync(d, nd, nv * sizeof(double), cudaMemcpyDeviceToDevice, S.stream); S.newton_accepted++; }
    }
    // :396-412 (rank == m here): NR / ProjPenalty with constraints, else YRetract with bounds, else Euclidean
    const int kind = (m > 0) ? ((!prm.do_project_retract && !(S.pinv_active && S.rank_cur < m)) ? 2 : 3) : (ineq ? 1 : 0);
    // armijo! (linesearch.jl:32-89)
    vec(S, nv, [=] __device__(int64_t i, double *acc) { acc[0] += d[i] * g[i]; }, 0, 1);
    finalize(S, 1u, 0);
    if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
    const double ar_dot = S.hctrl->s[0];
    double alpha = prm.alpha, newf = 0.0;
    f_diff = INFINITY; step_diff = INFINITY;
    int flag = 0;
    const double tl0 = now_ms();
    const bool exact = (prm.linesearch != 0 && !prm.disable_linesearch);                // :415-420
    if (exact) { if (exact_linesearch(c, S, kind, fval, &newf, &f_diff, &step_diff, &flag)) return S.cb_err ? LFPSQP_ERR_CALLBACK : LFPSQP_ERR_CUDA; }
    while (!exact && step_diff > prm.eps_x) {
      if (retract_trial(c, S, kind, alpha, &flag)) return S.cb_err ? LFPSQP_ERR_CALLBACK : LFPSQP_ERR_CUDA;
      // linesearch.jl:57-60 has no lower bound on alpha in this branch: when the retraction fails at EVERY alpha the
      // reference spins forever once alpha has underflowed to 0.  Stop at the floor the other branch uses (:82-85):
        // flag 98, LFPSQP_ST_NONFINITE.
      if (flag > 0) { if (alpha < 1e-100) { flag = 98; break; } alpha *= prm.s; continue; }   // :57-60
      fam_f(S, xnew);
      vec(S, n, [=] __device__(int64_t i, double *acc) { double t = xnew[i] - x[i]; acc[0] += t * t; }, 1, 1);   // slot 1 only
      finalize(S, 3u, 0);
      if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
      if (S.cb_err) return LFPSQP_ERR_CALLBACK;
      newf = S.hctrl->s[0];
      step_diff = sqrt(S.hctrl->s[1]);
      f_diff = fabs(newf - fval);
      if (prm.disable_linesearch) break;
      if ((newf - fval) <= prm.sigma * alpha * ar_dot) break;                           // :75
      alpha *= prm.s;
      if (alpha < 1e-100) { flag = 99; break; }
    }
    last_flag = flag;
    S.ms_linesearch += now_ms() - tl0;
    if (flag == 98) { status |= LFPSQP_ST_NONFINITE; cond = LFPSQP_MAX_ITER; break; }
    cudaMemcpyAsync(x, xnew, nv * sizeof(double), cudaMemcpyDeviceToDevice, S.stream);   // :424
    fval = newf;
    if (nobj < H) obj_hist[nobj] = fval;
    nobj++;
    it++;
    if (S.cb.callback && prm.callback_period > 0 && it % prm.callback_period == 0) {   // :432-434, param.callback(i, x)
      CK(cudaMemcpyAsync(S.hw, x, nv * sizeof(double), cudaMemcpyDeviceToHost, S.stream));
      CK(cudaStreamSynchronize(S.stream));
      if (S.cb.callback(S.cb.user, it, S.hw, nv)) return LFPSQP_ERR_CALLBACK;
    }
  }
  CK(cudaMemcpyAsync(x_out, x, n * sizeof(double), cudaMemcpyDeviceToHost, S.stream));
  if (m > 0) CK(cudaMemcpyAsync(lambda, S.lam, m * sizeof(double), cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  *obj_len = nobj;
  term->condition = cond; term->status = status; term->f_diff = f_diff; term->step_diff = step_diff;
  term->kkt_diff = kkt_diff; term->iter = it;
  if (stats) {
    stats->projcg_iters = S.projcg_iters; stats->projcg_negcurv = S.projcg_negcurv; stats->armijo_trials = S.armijo_trials;
    stats->retract_outer = S.retract_outer; stats->retract_pcg = S.retract_pcg; stats->pp_backtracks = S.pp_backtracks;
    stats->newton_accepted = S.newton_accepted; stats->factorizations = S.factorizations; stats->f_evals = S.f_evals;
    stats->flag_last = last_flag;
  }
  c->last_launches = S.launches;
  return LFPSQP_OK;
}

// ------------------------------------------------------------------ setup / teardown
void lfpsqp_large_release(lfpsqp_ctx *c) {
  if (!c->large) return;
  LargeState *S = c->large;
  cudaSetDevice(c->device);
  for (void *p : S->owned) cudaFree(p);
  if (S->hctrl) cudaFreeHost(S->hctrl);
  for (double *p : {S->hx, S->hv, S->hw, S->hlam, S->hc, S->hJ}) if (p) cudaFreeHost(p);
  if (S->side_stream) cudaStreamDestroy(S->side_stream);
  if (S->ev_panel) cudaEventDestroy(S->ev_panel);
  if (S->ev_potf) cudaEventDestroy(S->ev_potf);
  if (S->ev_g0) cudaEventDestroy(S->ev_g0);
  if (S->ev_g1) cudaEventDestroy(S->ev_g1);
  comm_release(*S);
  delete S;
  c->large = nullptr;
}

template <class T> static bool dalloc(LargeState &S, T **p, size_t count) {
  void *q = nullptr;
  if (cudaMalloc(&q, std::max<size_t>(count, 1) * sizeof(T)) != cudaSuccess) { cudaGetLastError(); return false; }
  S.owned.push_back(q); *p = (T *)q;
  return true;
}
// count = the number of ranks on which flag is set (one all-reduce: also a barrier of all ranks)
static int ranks_with(lfpsqp_ctx *c, LargeState &S, bool flag, int *count) {
  double v = flag ? 1.0 : 0.0;
  CK(cudaMemcpyAsync(S.commbuf, &v, 8, cudaMemcpyHostToDevice, S.stream));
  comm_allreduce(S, S.commbuf, 1);
  CK(cudaMemcpyAsync(&v, S.commbuf, 8, cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  *count = (int)lround(v);
  return 0;
}

extern "C" int lfpsqp_large_setup(lfpsqp_ctx *c, int family, int64_t n_global, int64_t m, int64_t col0, int64_t n_loc,
                                  const double *params, int params_on_device) {
  if (!c) return LFPSQP_ERR_ARG;
  cudaSetDevice(c->device);
  const bool csr = family == LFPSQP_FAM_SPARSE_QCQP_CSR;   // the same family with J kept sparse: S.family = SPARSE_QCQP, S.csr
  if (csr) family = LFPSQP_FAM_SPARSE_QCQP;
  if (family != LFPSQP_FAM_DIAGQUAD && family != LFPSQP_FAM_THOMSON && family != LFPSQP_FAM_HOST && family != LFPSQP_FAM_SPARSE_QCQP)
    return c->fail(LFPSQP_ERR_FAMILY, "large-n mode supports the DIAGQUAD, THOMSON, HOST (callback) and SPARSE_QCQP families");
  if (n_global < 1 || m < 0 || n_loc < 1 || col0 < 0 || col0 + n_loc > n_global || m > n_global)
    return c->fail(LFPSQP_ERR_ARG, "bad sizes for large-n setup");
  if (family == LFPSQP_FAM_SPARSE_QCQP && (n_loc != n_global || c->comm.world > 1))
    return c->fail(LFPSQP_ERR_FAMILY, "the SPARSE_QCQP family runs on one GPU (x'Qx couples column shards)");
  if (c->comm.world <= 1 && n_loc != n_global) return c->fail(LFPSQP_ERR_ARG, "a column shard needs a communicator (lfpsqp_comm_init)");
  if (family == LFPSQP_FAM_THOMSON && (n_global % 3 || m != n_global / 3 || n_loc % 3 || col0 % 3))
    return c->fail(LFPSQP_ERR_FAMILY, "THOMSON needs n = 3 m and column shards of whole points (col0 and n_loc multiples of 3)");
  if (m > 16384) return c->fail(LFPSQP_ERR_ARG, "m too large for the replicated factor");
  if (family == LFPSQP_FAM_HOST) {
    const lfpsqp_host_callbacks *cb = (const lfpsqp_host_callbacks *)params;
    if (!cb || !cb->f || !cb->grad || !cb->hess_lag_vec || (m > 0 && (!cb->c || !cb->jac)))
      return c->fail(LFPSQP_ERR_ARG, "HOST family: f, grad, hess_lag_vec (and c, jac when m > 0) callbacks are required");
    if (n_loc != n_global || c->comm.world > 1) return c->fail(LFPSQP_ERR_FAMILY, "the HOST (callback) family runs on one GPU");
  }
  SpqHost spq_host;   // validated and canonicalised before any previous state is released
  if (family == LFPSQP_FAM_SPARSE_QCQP) {
    if (!params) return c->fail(LFPSQP_ERR_ARG, "SPARSE_QCQP: params must point to a lfpsqp_sparse_qcqp descriptor");
    if (params_on_device) return c->fail(LFPSQP_ERR_ARG, "SPARSE_QCQP: the descriptor and its arrays are host memory (params_on_device must be 0)");
    int rc = spq_build(c, (const lfpsqp_sparse_qcqp *)params, n_global, m, spq_host);
    if (rc) return rc;
  }
  lfpsqp_large_release(c);
  LargeState *Sp = new LargeState(); LargeState &S = *Sp;
  c->large = Sp;
  S.comm = &c->comm; S.world = c->comm.world > 1 ? c->comm.world : 1; S.rank = c->comm.rank;
  S.family = family; S.csr = csr; S.n = n_global; S.n_loc = n_loc; S.nv = n_loc; S.col0 = col0; S.m = (int)m; S.stream = c->stream;
  S.sm_count = c->sm_count; S.ldj = up2(n_loc); S.ldm = up2(std::max<int64_t>(m, 1));
  S.vgrid = (int)std::min<int64_t>(std::max<int64_t>((n_loc + 255) / 256, 1), std::min<int64_t>(MAXP, 4 * (int64_t)c->sm_count));
  S.np_loop_raw = S.vgrid; S.np_loop = (S.world > 1) ? 1 : S.vgrid;
  // row splits of pass 2: enough CTAs to fill the GPU, at least 32 rows per split
  {
    int64_t coltiles = (n_loc + 511) / 512;
    int want = (int)std::max<int64_t>(1, (4LL * c->sm_count + coltiles - 1) / coltiles);
    int maxs = std::max(1, (int)m / 32);
    S.nsplit = std::max(1, std::min(std::min(want, maxs), 64));
    S.rows_per_split = m > 0 ? (int)((m + S.nsplit - 1) / S.nsplit) : 1;
    S.nsplit = m > 0 ? (int)((m + S.rows_per_split - 1) / S.rows_per_split) : 1;
  }
  S.jsplit = csr ? 1 : S.nsplit;
  S.cg_chunk = 2; S.pcg_chunk = 2;
  const size_t nl = (size_t)n_loc, mm = (size_t)std::max<int64_t>(m, 1);
  bool ok = true;
  if (!csr) ok &= dalloc(S, &S.J, mm * S.ldj);
  ok &= dalloc(S, &S.G, mm * S.ldm); ok &= dalloc(S, &S.XT, mm * S.ldm); ok &= dalloc(S, &S.Linv, mm * S.ldm);
  ok &= dalloc(S, &S.Dblk, ((mm + 63) / 64) * 64 * 64); ok &= dalloc(S, &S.tmp64, mm * 64); ok &= dalloc(S, &S.thresh, 8);
  S.nz_rows = (int)((mm + 63) / 64); S.nz_ld = (int64_t)((S.ldj + GM_BK - 1) / GM_BK + 64) / 64 * 64; S.gram_mode = 0; S.nz_pending = false; S.g_blockdiag = 0; S.gdep_pending = false;
  if (!csr) ok &= dalloc(S, &S.nzmap, (size_t)S.nz_rows * S.nz_ld);
  ok &= dalloc(S, &S.blkflag, (size_t)S.nz_rows * S.nz_rows + S.nz_rows + 1);   // + done[nblk]
  ok &= dalloc(S, &S.invflag, (size_t)S.nz_rows * S.nz_rows + 1);
  { int dev = 0, v = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev); if (v > 2048) S.max_dyn_smem = v - 1024; }
  S.gemm_ws_bytes = std::max<size_t>((size_t)16 * mm * 64 * 8, std::min<size_t>(mm * mm * 8 * 16, (size_t)1 << 30));
  { char *ws = nullptr; ok &= dalloc(S, &ws, S.gemm_ws_bytes); S.gemm_ws = (double *)ws; }
  double **vecs[] = {&S.x, &S.xnew, &S.xtil, &S.g, &S.d, &S.nd, &S.w0, &S.w1, &S.w2, &S.w3, &S.w4, &S.hdiag};
  for (double **v : vecs) ok &= dalloc(S, v, 2 * nl + 2);   // [x-half | y-half] when bounds are set later
  double **mv[] = {&S.cval, &S.lam, &S.tm, &S.ty, &S.tu, &S.nr_t1, &S.nr_t2, &S.nr_dc, &S.cvc};
  for (double **v : mv) ok &= dalloc(S, v, mm + 2);
  ok &= dalloc(S, &S.cpart, (size_t)S.nsplit * std::max(nl, mm) + 2);
  ok &= dalloc(S, &S.lp, (size_t)NSLOT * MAXP); ok &= dalloc(S, &S.gpart, (size_t)NSLOT * MAXP);
  ok &= dalloc(S, &S.ctrl, 1); ok &= dalloc(S, &S.commbuf, 64);
  if (family == LFPSQP_FAM_THOMSON) {
    ok &= dalloc(S, &S.pairws, (size_t)16 * nl + 2);
    if (S.world > 1) { ok &= dalloc(S, &S.xfull, (size_t)n_global + 2); ok &= dalloc(S, &S.xfull_h, (size_t)n_global + 2); ok &= dalloc(S, &S.vfull, (size_t)n_global + 2); }
  }
  S.Dnr = nullptr;
  if (family == LFPSQP_FAM_HOST) {
    S.cb = *(const lfpsqp_host_callbacks *)params;
    ok &= dalloc(S, &S.Jstage, mm * nl);
    bool hok = cudaMallocHost((void **)&S.hx, (nl + 2) * 8) == cudaSuccess && cudaMallocHost((void **)&S.hv, (2 * nl + 2) * 8) == cudaSuccess &&
               cudaMallocHost((void **)&S.hw, (2 * nl + 2) * 8) == cudaSuccess && cudaMallocHost((void **)&S.hlam, (mm + 2) * 8) == cudaSuccess &&
               cudaMallocHost((void **)&S.hc, (mm + 2) * 8) == cudaSuccess && cudaMallocHost((void **)&S.hJ, mm * nl * 8) == cudaSuccess;
    if (!hok) { cudaGetLastError(); ok = false; }
  }
  if (!ok) { lfpsqp_large_release(c); return c->fail(LFPSQP_ERR_NOMEM, "large-n setup: device allocation failed"); }
  if (cudaMallocHost((void **)&S.hctrl, sizeof(LargeCtrl)) != cudaSuccess) { lfpsqp_large_release(c); return c->fail(LFPSQP_ERR_NOMEM, "pinned allocation failed"); }
  cudaEventCreate(&S.ev_g0); cudaEventCreate(&S.ev_g1);
  cudaMemsetAsync(S.lp, 0, (size_t)NSLOT * MAXP * 8, S.stream); cudaMemsetAsync(S.gpart, 0, (size_t)NSLOT * MAXP * 8, S.stream);
  cudaMemsetAsync(S.ctrl, 0, sizeof(LargeCtrl), S.stream);
  if (S.J) cudaMemsetAsync(S.J, 0, mm * S.ldj * sizeof(double), S.stream);   // the pad column of an odd n_loc must stay zero (16-byte K chunks)
  // parameters
  if (family == LFPSQP_FAM_DIAGQUAD) {
    const size_t cnt = 2 * mm * nl * (m > 0 ? 1 : 0) + (size_t)m + 2 * nl;
    if (!params) { lfpsqp_large_release(c); return c->fail(LFPSQP_ERR_ARG, "DIAGQUAD needs a parameter blob"); }
    if (S.ldj != n_loc) { lfpsqp_large_release(c); return c->fail(LFPSQP_ERR_ARG, "large-n mode needs an even local column count"); }
    const double *blob = params;
    if (!params_on_device) {
      double *dev = nullptr;
      if (!dalloc(S, &dev, cnt)) { lfpsqp_large_release(c); return c->fail(LFPSQP_ERR_NOMEM, "parameter allocation failed"); }
      CK(cudaMemcpyAsync(dev, params, cnt * 8, cudaMemcpyHostToDevice, S.stream));
      blob = dev;
    }
    S.p_Q = blob; S.p_A = blob + (size_t)m * nl; S.p_b = S.p_A + (size_t)m * nl; S.p_xt = S.p_b + m; S.p_w = S.p_xt + nl;
    if ((((uintptr_t)S.p_A) & 15) || (((uintptr_t)S.p_Q) & 15)) { lfpsqp_large_release(c); return c->fail(LFPSQP_ERR_ARG, "parameter blob must be 16-byte aligned"); }
  }
  if (family == LFPSQP_FAM_SPARSE_QCQP && (!spq_upload(S, spq_host) || (csr && !spj_upload(S, spq_host)))) {
    lfpsqp_large_release(c);
    return c->fail(LFPSQP_ERR_NOMEM, "SPARSE_QCQP: device allocation or upload of the structures failed");
  }
  cudaFuncSetAttribute(dgemm_nt_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dgemm_smem_bytes<128>());
  cudaFuncSetAttribute(dgemm_nt_kernel<128, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dgemm_smem_bytes<128>());
  cudaFuncSetAttribute(dgemm_nt_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dgemm_smem_bytes<64>());
  { int dev = 0, v = 0; cudaGetDevice(&dev); cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
    if (v > 2048) CK(cudaFuncSetAttribute(dgemm_nt_kernel<128, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, v - 1024)); }   // static shared memory counts too
  cudaFuncSetAttribute(potf2_inv_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * 64 * 65 * sizeof(double)));
  cudaFuncSetAttribute(potf2_inv_indep_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(2 * 64 * 65 * sizeof(double)));
  // the staged m-vector of tri_gemv / the row-split of cols_dot exceed the 48 KB default for m > 6144
  CK(cudaFuncSetAttribute(tri_gemv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(mm * sizeof(double), 1024)));
  CK(cudaFuncSetAttribute(cols_dot_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(mm * sizeof(double), 1024)));
  CK(cudaFuncSetAttribute(cols_dot_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(mm * sizeof(double), 1024)));
  if (csr) {   // the shared m-vector of the sparse Gram (128 KB at m = 16384)
    CK(cudaFuncSetAttribute(spj_gram_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(mm * sizeof(double), 1024)));
    CK(cudaFuncSetAttribute(spj_gram_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(mm * sizeof(double), 1024)));
  }
  CK(cudaStreamSynchronize(S.stream));
  // the environment switches of the README (A/B measurements, tests), read once per problem
  const char *fused_env = getenv("LFPSQP_FUSED_PROJCG"), *skip_env = getenv("LFPSQP_GRAM_SKIP"), *inv_env = getenv("LFPSQP_EXPLICIT_INVERSE");
  S.gram_skip = !(skip_env && skip_env[0] == '0');
  S.force_inverse = (inv_env && (inv_env[0] == '0' || inv_env[0] == '1')) ? inv_env[0] - '0' : -1;
  // pcg! is fused for every family with a dense J, projcg for diagonal Hessians; the CSR form runs the launch-per-phase loops
  if (m > 0 && !csr && !(fused_env && fused_env[0] == '0')) fused_projcg_init(S, c->device);
  if (S.world > 1) {
    // every rank must take the same path (a rank in the launch-per-phase loop would deadlock against peers inside the fused
    // mailbox protocol): fused only if ALL ranks are eligible.  The all-reduce is also the barrier that ends setup, so that
    // no rank starts exchanging while another one is still uploading its parameters.
    int fused_ranks = 0;
    int rc = ranks_with(c, S, S.fused_ok, &fused_ranks);
    if (rc) return rc;
    if (fused_ranks < S.world) S.fused_ok = false;
  }
  return LFPSQP_OK;
}

static int need_large(lfpsqp_ctx *c) {
  if (!c) return LFPSQP_ERR_ARG;
  if (!c->large) return c->fail(LFPSQP_ERR_ARG, "call lfpsqp_large_setup first");
  cudaSetDevice(c->device);
  c->large->stream = c->stream;
  std::fill(c->large->disp, c->large->disp + 8, (int64_t)0);   // every entry call starts a new dispatch record
  return 0;
}
// need_large for the unit-level ops: with bounds they work on one GPU only (a column shard's embedding rows are not exchanged)
static int need_unit(lfpsqp_ctx *c) {
  int rc = need_large(c); if (rc) return rc;
  if (c->large->ineq && c->large->world > 1)
    return c->fail(LFPSQP_ERR_UNSUPPORTED, "unit-level large-n ops with bounds run on one GPU (this problem is column-sharded)");
  return 0;
}
static int prep_params(lfpsqp_ctx *c, LargeState &S, const lfpsqp_params *prm) {
  if (!prm) return c->fail(LFPSQP_ERR_ARG, "params is NULL");
  if (prm->beta > 0 && !S.cb.randn) {
    if (!c->noise_host) return c->fail(LFPSQP_ERR_UNSUPPORTED, "beta>0 needs the caller's noise: lfpsqp_ctx_set_noise (device families) or the randn host callback (LFPSQP_FAM_HOST)");
    if (c->noise_N != S.nv || c->noise_B != 1) return c->fail(LFPSQP_ERR_ARG, "lfpsqp_ctx_set_noise: large-n mode needs B = 1 and rows of %lld entries (this rank's working entries)", (long long)S.nv);
    if (S.noise_cap < (size_t)c->noise_T * S.nv) {
      if (!dalloc(S, &S.noise_dev, (size_t)c->noise_T * S.nv)) return c->fail(LFPSQP_ERR_NOMEM, "noise buffer allocation failed");
      S.noise_cap = (size_t)c->noise_T * S.nv;
    }
    CK(cudaMemcpyAsync(S.noise_dev, c->noise_host, (size_t)c->noise_T * S.nv * 8, cudaMemcpyHostToDevice, S.stream));
    S.noise_T = c->noise_T;
  } else S.noise_T = 0;
  S.prm = *prm;
  if (prm->linesearch != 0 && !prm->disable_linesearch && !S.ex[0]) {
    for (int i = 0; i < 4; i++) if (!dalloc(S, &S.ex[i], 2 * (size_t)S.n_loc + 2)) return c->fail(LFPSQP_ERR_NOMEM, "exact line search workspace allocation failed");
  }
  if (!prm->do_project_retract && S.m > 0 && !S.Dnr) {
    if (!dalloc(S, &S.Dnr, (size_t)S.m * S.ldm)) return c->fail(LFPSQP_ERR_NOMEM, "NR workspace allocation failed");
  }
  return 0;
}

extern "C" int lfpsqp_large_solve(lfpsqp_ctx *c, const double *x0_loc, const lfpsqp_params *prm, double *x_out_loc,
                                  double *obj_hist, int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term,
                                  lfpsqp_stats *stats) {
  int rc = need_large(c); if (rc) return rc;
  LargeState &S = *c->large;
  rc = prep_params(c, S, prm); if (rc) return rc;
  if (H < 1) return c->fail(LFPSQP_ERR_ARG, "H must be >= 1");
  cudaEventRecord(c->ev0, S.stream);
  rc = solve(c, S, x0_loc, x_out_loc, obj_hist, H, obj_len, lambda, term, stats);
  if (rc) return S.hctrl->commfail ? LFPSQP_ERR_COMM : rc;
  cudaEventRecord(c->ev1, S.stream);
  cudaEventSynchronize(c->ev1);
  float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms;
  return LFPSQP_OK;
}

int build_bounds_public(int64_t n, int64_t p, const double *xl, const double *xu, std::vector<double> &bnd);  // abi.cu

// Bounds of this rank's entries: InequalityData (src/inequality_helper.jl:39-85) + the workspaces of the 2n embedding.
extern "C" int lfpsqp_large_set_bounds(lfpsqp_ctx *c, const double *xl_loc, const double *xu_loc) {
  int rc = need_large(c); if (rc) return rc;
  LargeState &S = *c->large;
  const int64_t nl = S.n_loc;
  std::vector<double> bnd;
  int ineq = build_bounds_public(nl, 0, xl_loc, xu_loc, bnd);
  if (ineq == LFPSQP_ERR_BOUNDS) return c->fail(LFPSQP_ERR_BOUNDS, "Infeasible: lower bounds cannot be greater than upper bounds");
  if (ineq < 0) return c->fail(LFPSQP_ERR_ARG, "xl and xu must both be given or both be NULL");
  if (S.world > 1) {  // optimize.jl:151 looks at ALL of xl, xu: any rank with a finite bound switches every rank
    int bounded_ranks = 0;
    if ((rc = ranks_with(c, S, ineq != 0, &bounded_ranks))) return rc;
    if (bounded_ranks > 0 && !ineq) bnd.assign(5 * nl, 0.0);   // this shard: all lines (q = r = s = t = 0)
    ineq = bounded_ranks > 0;
  }
  S.ineq = ineq != 0;
  S.nv = S.ineq ? 2 * nl : nl;
  if (!S.ineq) return LFPSQP_OK;   // S.I keeps its workspaces: bounds may be switched on again later
  if (!S.bq) {
    bool ok = true;
    double **nvv[] = {&S.bq, &S.br, &S.bs, &S.bt, &S.I.Dx, &S.I.Dy, &S.I.S, &S.I.lamy, &S.cvh, &S.pb};
    for (double **v : nvv) ok &= dalloc(S, v, (size_t)nl + 2);
    if (S.m > 0 && !S.csr) { ok &= dalloc(S, &S.Jw, (size_t)S.m * S.ldj); if (ok) cudaMemsetAsync(S.Jw, 0, (size_t)S.m * S.ldj * 8, S.stream); }
    if (!ok) return c->fail(LFPSQP_ERR_NOMEM, "bound-embedding workspace allocation failed");
  }
  // bnd layout (abi.cu build_bounds): [kind | q | r | s | t], each nl doubles
  CK(cudaMemcpyAsync(S.bq, bnd.data() + nl, nl * 8, cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemcpyAsync(S.br, bnd.data() + 2 * nl, nl * 8, cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemcpyAsync(S.bs, bnd.data() + 3 * nl, nl * 8, cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemcpyAsync(S.bt, bnd.data() + 4 * nl, nl * 8, cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemsetAsync(S.I.lamy, 0, nl * 8, S.stream));
  CK(cudaStreamSynchronize(S.stream));   // bnd is a stack-owned host vector
  S.I.q = S.bq; S.I.r = S.br; S.I.s = S.bs; S.I.t = S.bt; S.I.nx = nl;
  if (S.world > 1) {   // leave together: nobody starts a solve while a peer is still uploading its bound tables
    comm_allreduce(S, S.commbuf, 1);
    CK(cudaStreamSynchronize(S.stream));
  }
  return LFPSQP_OK;
}

// optimize(...) for one large instance on one GPU with host-resident family parameters
extern "C" int lfpsqp_solve_large(lfpsqp_ctx *c, int family, int64_t n, int64_t m, const double *fam_params,
                                  const double *x0, const double *xl, const double *xu, const lfpsqp_params *prm,
                                  double *x_out, double *obj_hist, int64_t H, int64_t *obj_len, double *lambda,
                                  lfpsqp_term *term, lfpsqp_stats *stats) {
  if (!c) return LFPSQP_ERR_ARG;
  int rc = lfpsqp_large_setup(c, family, n, m, 0, n, fam_params, 0);
  if (rc) return rc;
  rc = lfpsqp_large_set_bounds(c, xl, xu);
  if (rc) return rc;
  return lfpsqp_large_solve(c, x0, prm, x_out, obj_hist, H, obj_len, lambda, term, stats);
}

// The explicit-derivative core optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m, param) (src/optimize.jl:119-443) for
// an arbitrary problem whose callbacks run on the host; all linear algebra of the hot path runs on the device.
extern "C" int lfpsqp_solve_host(lfpsqp_ctx *c, const lfpsqp_host_callbacks *cb, int64_t n, int64_t m, const double *x0,
                                 const double *xl, const double *xu, const lfpsqp_params *prm, double *x_out,
                                 double *obj_hist, int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term,
                                 lfpsqp_stats *stats) {
  return lfpsqp_solve_large(c, LFPSQP_FAM_HOST, n, m, (const double *)cb, x0, xl, xu, prm, x_out, obj_hist, H, obj_len, lambda,
                            term, stats);
}

// Unit-level: factorisation of the Jacobian at x (ksvd! replacement) -- G = J J' (lower), L, L^-1 returned to the host.
// With bounds x is the working point [x | y] (2 n_loc entries) and G is the weighted G_w = J diag(Dy^2) J' of that point.
extern "C" int lfpsqp_large_factor(lfpsqp_ctx *c, const double *x_loc, double *G_out, double *L_out, double *Linv_out,
                                   int *rank_deficient, double *gram_ms) {
  int rc = need_unit(c); if (rc) return rc;
  LargeState &S = *c->large;
  lfpsqp_params p; lfpsqp_default_params(&p); S.prm = p;
  const int m = S.m; const size_t ldm = S.ldm;
  CK(cudaMemcpyAsync(S.x, x_loc, S.nv * 8, cudaMemcpyHostToDevice, S.stream));
  reset_ctrl(S);
  if (S.ineq) ineq_gradient(S, S.x);   // Dx, Dy, S of the point: the weights of G_w and the bound part of the projector (:277)
  if (m < 1) {   // nothing to factorise; with bounds the projector is the bound part alone
    CK(cudaStreamSynchronize(S.stream));
    if (rank_deficient) *rank_deficient = 0;
    if (gram_ms) *gram_ms = 0.0;
    return LFPSQP_OK;
  }
  fam_c_jac(S, true, S.cval, S.x);
  gram(S, true);
  if (G_out) CK(cudaMemcpy2DAsync(G_out, m * 8, S.G, ldm * 8, m * 8, m, cudaMemcpyDeviceToHost, S.stream));   // before L overwrites it
  S.prefer_pinv = false;
  factorize(c, S);
  if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
  const int lost_rank = S.hctrl->rankflag;
  if (lost_rank) {   // truncated path: the later project / projcg calls use the pseudo-inverse; L / L^-1 are not defined
    S.hctrl->rankflag = 0; write_ctrl_fields(S);
    if (factorize_pinv(c, S, true)) return LFPSQP_ERR_CUDA;
    if (read_ctrl(c, S)) return LFPSQP_ERR_CUDA;
    S.rank_cur = (int)S.hctrl->s[14];
    S.prefer_pinv = false;
  }
  if (L_out) CK(cudaMemcpy2DAsync(L_out, m * 8, S.G, ldm * 8, m * 8, m, cudaMemcpyDeviceToHost, S.stream));
  if (Linv_out) CK(cudaMemcpy2DAsync(Linv_out, m * 8, S.Linv, ldm * 8, m * 8, m, cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  if (rank_deficient) *rank_deficient = lost_rank ? (m - S.rank_cur > 0 ? m - S.rank_cur : 1) : 0;   // 0, or the rank defect found
  if (gram_ms) { float ms = 0; cudaEventElapsedTime(&ms, S.ev_g0, S.ev_g1); *gram_ms = ms; }
  return LFPSQP_OK;
}

// Unit-level: tangent projection v - J'(J J')^-1 J v with the factor cached by lfpsqp_large_factor (kgemv! pair,
// optimize.jl:306-307) and the multipliers (J J')^-1 J v (optimize.jl:333-343).  With bounds v is a working vector
// (2 n_loc entries), the projector is the one of the 2n embedding at the factorised point and lambda_out receives
// [lambda (m) ; lambda_y (n_loc)] (calculate_lambda_kkt!, inequality_helper.jl:286-308).
extern "C" int lfpsqp_large_project(lfpsqp_ctx *c, const double *v_loc, double *v_out_loc, double *lambda_out) {
  int rc = need_unit(c); if (rc) return rc;
  LargeState &S = *c->large;
  CK(cudaMemcpyAsync(S.d, v_loc, S.nv * 8, cudaMemcpyHostToDevice, S.stream));
  project(S, S.d, S.lam, 0, 0, /*want_mult=*/1);
  CK(cudaMemcpyAsync(v_out_loc, S.d, S.nv * 8, cudaMemcpyDeviceToHost, S.stream));
  if (lambda_out && S.m > 0) CK(cudaMemcpyAsync(lambda_out, S.lam, S.m * 8, cudaMemcpyDeviceToHost, S.stream));
  if (lambda_out && S.ineq) CK(cudaMemcpyAsync(lambda_out + S.m, S.I.lamy, S.n_loc * 8, cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  return LFPSQP_OK;
}

// Unit-level + benchmark: projcg! (projcg.jl:40-121) at the point x with multipliers lam, right-hand side b = P(-grad f(x)),
// tolerance tol, at most maxit iterations (tol = 0 with maxit = K times a fixed number of iterations: the
// "projcg iterations / s" metric).  Needs lfpsqp_large_factor at the same x first.  ms = device time of the loop.
// With bounds x and the solution are working vectors (2 n_loc entries), lam is [lambda (m) ; lambda_y (n_loc)] and the
// Hessian is the augmented one of inequality_helper.jl:144-158.
extern "C" int lfpsqp_large_projcg(lfpsqp_ctx *c, const double *x_loc, const double *lam, double tol, int64_t maxit,
                                   int chunk, double *sol_out_loc, int64_t *iters, double *nr, int *status, double *ms) {
  int rc = need_unit(c); if (rc) return rc;
  LargeState &S = *c->large;
  const int64_t n = S.nv;
  double *g = S.g, *d = S.d;
  CK(cudaMemcpyAsync(S.x, x_loc, n * 8, cudaMemcpyHostToDevice, S.stream));
  if (S.m > 0) { if (lam) CK(cudaMemcpyAsync(S.lam, lam, S.m * 8, cudaMemcpyHostToDevice, S.stream)); else cudaMemsetAsync(S.lam, 0, S.m * 8, S.stream); }
  if (S.ineq) {   // lambda_y of the Hessian; g has a zero y-half (optimize.jl:191)
    if (lam) CK(cudaMemcpyAsync(S.I.lamy, lam + S.m, S.n_loc * 8, cudaMemcpyHostToDevice, S.stream));
    else CK(cudaMemsetAsync(S.I.lamy, 0, S.n_loc * 8, S.stream));
    CK(cudaMemsetAsync(g + S.n_loc, 0, S.n_loc * 8, S.stream));
  }
  reset_ctrl(S);
  if (S.ineq) ineq_gradient(S, S.x);
  fam_grad(S, g, S.x);
  vec(S, n, [=] __device__(int64_t i, double *) { d[i] = -1.0 * g[i]; });
  if (S.m > 0 || S.ineq) project(S, d, nullptr, 0, 0);
  fam_hess_prepare(S, S.x, S.lam);
  S.reset_counters();
  cudaEventRecord(c->ev0, S.stream);
  if (projcg(c, S, tol, maxit, chunk > 0 ? chunk : S.cg_chunk)) return LFPSQP_ERR_CUDA;
  cudaEventRecord(c->ev1, S.stream);
  if (sol_out_loc) CK(cudaMemcpyAsync(sol_out_loc, S.nd, n * 8, cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  float t = 0; cudaEventElapsedTime(&t, c->ev0, c->ev1);
  if (ms) *ms = t;
  if (iters) *iters = S.hctrl->iter;
  if (nr) *nr = S.hctrl->nr;
  if (status) *status = S.hctrl->status;
  c->last_ms = t; c->last_launches = S.launches;
  return LFPSQP_OK;
}

// Unit-level: the general projcg!(x, lambda, A, U, b, c; tol, maxit) of src/projcg.jl:40-121 (test/test_cg.jl:10-28 uses c != 0):
// A = Lagrangian Hessian of the family at (x_point, lam), U = orthonormal Cholesky-QR basis J(x_point)' L^-T of the range of
// J', b (n_loc) and c (m) given by the caller.  Needs lfpsqp_large_factor at x_point first.  Runs the launch-per-phase loop.
extern "C" int lfpsqp_large_projcg_general(lfpsqp_ctx *c, const double *x_loc, const double *lam, const double *b_loc,
                                           const double *cvec, double tol, int64_t maxit, double *sol_out_loc,
                                           double *lambda_out, int64_t *iters, double *nr, int *status) {
  int rc = need_unit(c); if (rc) return rc;
  LargeState &S = *c->large;
  if (S.ineq) return c->fail(LFPSQP_ERR_UNSUPPORTED, "projcg_general works on the unbounded problem: its start x0 = U c and its multipliers U'(b - A x) have no bound-embedding form here");
  if (!x_loc || !b_loc) return c->fail(LFPSQP_ERR_ARG, "x and b are required");
  const int64_t n = S.n_loc;
  CK(cudaMemcpyAsync(S.x, x_loc, n * 8, cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemcpyAsync(S.d, b_loc, n * 8, cudaMemcpyHostToDevice, S.stream));
  if (S.m > 0) { if (lam) CK(cudaMemcpyAsync(S.lam, lam, S.m * 8, cudaMemcpyHostToDevice, S.stream)); else cudaMemsetAsync(S.lam, 0, S.m * 8, S.stream); }
  if (S.m > 0 && cvec) CK(cudaMemcpyAsync(S.nr_t1, cvec, S.m * 8, cudaMemcpyHostToDevice, S.stream));
  reset_ctrl(S);
  fam_hess_prepare(S, S.x, S.lam);
  S.reset_counters();
  if (projcg(c, S, tol, maxit, S.cg_chunk, (S.m > 0 && cvec) ? S.nr_t1 : nullptr, (S.m > 0 && lambda_out) ? S.nr_t2 : nullptr)) return LFPSQP_ERR_CUDA;
  const int st = S.hctrl->status; const int64_t it = S.hctrl->iter; const double nrv = S.hctrl->nr;
  if (sol_out_loc) CK(cudaMemcpyAsync(sol_out_loc, S.nd, n * 8, cudaMemcpyDeviceToHost, S.stream));
  if (lambda_out && S.m > 0) CK(cudaMemcpyAsync(lambda_out, S.nr_t2, S.m * 8, cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  if (iters) *iters = it;
  if (nr) *nr = nrv;
  if (status) *status = st;
  c->last_launches = S.launches;
  return LFPSQP_OK;
}

// Unit-level: retract!(cval, xnew, c!, xtilde, x, method) (src/retractions.jl:75-177 NR / :265-441 ProjPenalty) with the
// factorisation taken at x_base (as armijo! calls it, linesearch.jl:52).  method: 0 = NR, 1 = ProjPenalty.  With bounds
// x_base, xtilde and xnew are working points [x | y] (2 n_loc entries), and the c-part of ProjPenalty's merit vector
// starts at zero, as at the start of a solve.
extern "C" int lfpsqp_large_retract(lfpsqp_ctx *c, int method, const double *x_base_loc, const double *xtilde_loc,
                                    const lfpsqp_params *prm, double *xnew_out_loc, double *cval_out, int *flag,
                                    int64_t *iters, int64_t *pcg_iters) {
  int rc = need_unit(c); if (rc) return rc;
  LargeState &S = *c->large;
  lfpsqp_params p2 = *prm; p2.do_project_retract = (method == 0) ? 0 : 1;
  rc = prep_params(c, S, &p2); if (rc) return rc;
  if (S.m < 1) return c->fail(LFPSQP_ERR_ARG, "retraction needs m > 0");
  const int64_t n = S.nv;
  CK(cudaMemcpyAsync(S.x, x_base_loc, n * 8, cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemcpyAsync(S.xtil, xtilde_loc, n * 8, cudaMemcpyHostToDevice, S.stream));
  if (S.ineq) CK(cudaMemsetAsync(S.cvc, 0, S.m * 8, S.stream));
  reset_ctrl(S);
  S.reset_counters();
  if (S.ineq) ineq_gradient(S, S.x);
  fam_c_jac(S, true, S.cval, S.x);
  gram(S, true);
  if (factorize(c, S)) return LFPSQP_ERR_CUDA;
  int fl = 0, i1 = 0, i2 = 0;
  if (method == 0) { if (retract_nr(c, S, &fl, &i1)) return LFPSQP_ERR_CUDA; }
  else { if (retract_pp(c, S, &fl, &i1, &i2)) return LFPSQP_ERR_CUDA; }
  CK(cudaMemcpyAsync(xnew_out_loc, S.xnew, n * 8, cudaMemcpyDeviceToHost, S.stream));
  if (cval_out) CK(cudaMemcpyAsync(cval_out, S.cval, S.m * 8, cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  if (flag) *flag = fl; if (iters) *iters = i1; if (pcg_iters) *pcg_iters = i2;
  c->last_launches = S.launches;
  return LFPSQP_OK;
}

// Unit-level: pcg!(mu, J, no_precondition, x, r, p, z, tmp_m, tol, maxiter) (src/retractions.jl:179-246) with J = jac(x_point),
// x = 0, r = b.  Outputs the solution, the final residual, flag (1 iff iters == maxiter) and the iteration count.  With
// bounds x_point, b and the outputs are working vectors (2 n_loc entries) and the operator is bigA bigA' + mu I at x_point.
extern "C" int lfpsqp_large_pcg(lfpsqp_ctx *c, const double *x_point_loc, double mu, const double *b_loc, double tol,
                                int64_t maxiter, double *x_out_loc, double *r_out_loc, int *flag, int64_t *iters) {
  int rc = need_unit(c); if (rc) return rc;
  LargeState &S = *c->large;
  if (S.m < 1) return c->fail(LFPSQP_ERR_ARG, "pcg needs m > 0");
  const int64_t n = S.nv;
  double *r = S.w0, *pv = S.w1, *dx = S.w3, *lp = S.lp;
  CK(cudaMemcpyAsync(S.x, x_point_loc, n * 8, cudaMemcpyHostToDevice, S.stream));
  CK(cudaMemcpyAsync(r, b_loc, n * 8, cudaMemcpyHostToDevice, S.stream));
  reset_ctrl(S);
  S.reset_counters();
  if (S.ineq) ineq_gradient(S, S.x);   // Dx, Dy, S of bigA at x_point
  fam_c_jac(S, true, S.cval, S.x);
  pcg_start_kernel<<<S.vgrid, 256, 0, S.stream>>>(n, r, dx, pv, lp);
  cudaEventRecord(c->ev0, S.stream);
  if (run_pcg(c, S, mu, tol, maxiter)) return LFPSQP_ERR_CUDA;
  cudaEventRecord(c->ev1, S.stream);
  if (x_out_loc) CK(cudaMemcpyAsync(x_out_loc, dx, n * 8, cudaMemcpyDeviceToHost, S.stream));
  if (r_out_loc) CK(cudaMemcpyAsync(r_out_loc, r, n * 8, cudaMemcpyDeviceToHost, S.stream));
  CK(cudaStreamSynchronize(S.stream));
  if (iters) *iters = S.hctrl->pcg_iter;
  if (flag) *flag = (S.hctrl->pcg_iter == maxiter) ? 1 : 0;
  { float ms = 0; cudaEventElapsedTime(&ms, c->ev0, c->ev1); c->last_ms = ms; }   // device time of the pcg! loop (lfpsqp_last_kernel_ms)
  c->last_launches = S.launches;
  return LFPSQP_OK;
}

// length of this rank's working vectors: n_loc, or 2 n_loc once lfpsqp_large_set_bounds has switched the embedding on
extern "C" int lfpsqp_large_working_length(lfpsqp_ctx *c, int64_t *nv) {
  if (!c || !c->large || !nv) return LFPSQP_ERR_ARG;
  *nv = c->large->nv;
  return LFPSQP_OK;
}

// what the last large-n entry call enqueued (LargeState::disp, large_state.h): read-only, recorded on the host
extern "C" int lfpsqp_large_last_dispatch(lfpsqp_ctx *c, int64_t *out8) {
  if (!c || !c->large || !out8) return LFPSQP_ERR_ARG;
  std::copy(c->large->disp, c->large->disp + 8, out8);
  return LFPSQP_OK;
}

// host wall-clock split of the last lfpsqp_large_solve (every phase starts and ends at a host<->device sync):
// out = [factorisation incl. jac!/Gram/Cholesky/first projection, projcg!, line search incl. retractions, total device ms]
extern "C" int lfpsqp_large_phase_ms(lfpsqp_ctx *c, double *out4) {
  if (!c || !c->large || !out4) return LFPSQP_ERR_ARG;
  out4[0] = c->large->ms_factor; out4[1] = c->large->ms_projcg; out4[2] = c->large->ms_linesearch; out4[3] = c->last_ms;
  return LFPSQP_OK;
}
