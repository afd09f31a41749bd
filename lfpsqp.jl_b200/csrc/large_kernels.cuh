// large_kernels.cuh -- streaming (HBM-bound) kernels of the large-n mode.
//
//   rows_dot      t = J v          pass 1 of the tangent projection / of pcg!'s J'(J p)   (projcg.jl:96, retractions.jl:221)
//   cols_dot      J' u             pass 2                                                   (projcg.jl:97, retractions.jl:222)
//   tri_gemv      y = L^-1 t, u = L^-T y   (replaces U'(.) / Sigma^-1 V' of the SVD path, SURVEY.md App. B)
//   cg_* / pcg_*  fused vector updates + dot-product partials of projcg! (projcg.jl:71-112) and pcg! (retractions.jl:207-238)
//
// J is m x n_loc ROW-major (== the reference's Jct, optimize.jl:190): rows_dot streams rows with 128-bit loads,
// cols_dot streams the same rows with threads mapped to columns.  Algorithmic bytes per projcg iteration:
// 16*m*N (two passes over J) + 8*m^2 (two triangular GEMVs) + ~104*N (vector sweeps)  (SURVEY.md 8d).
// All dot products are two-level deterministic reductions (per-CTA partials, fixed-order final sum): no atomics.
// Every kernel of an iteration is predicated on ctrl->status so that the host can enqueue iterations in chunks
// (or as a CUDA graph) and look at the status only once per chunk.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include "large_ctrl.h"
#include "large_device.cuh"

namespace lfpsqp {

// ------------------------------------------------------------------ pass 1: t[i] = sum_j J[i][j] v[j]
// One CTA owns R full rows (no cross-CTA reduction). v is re-read from L2 once per R rows.
// SKIP: nz is the zero-slab map of J (large_gemm.cuh::zero_slab_map_kernel: 64 rows x 16 columns); loads of all-zero slabs are
// not issued.  Same threads, same accumulation order, only "+ 0 * v" terms less: bit-identical to the dense pass.
template <int R, bool SKIP = false>
__global__ void __launch_bounds__(256) rows_dot_kernel(const double *__restrict__ J, int64_t ld, int m, int64_t ncols,
                                                       const double *__restrict__ v, double *__restrict__ t,
                                                       const LargeCtrl *ctrl, int pred, const unsigned char *__restrict__ nz = nullptr,
                                                       int64_t nz_ld = 0) {
  if (pred == 1 && ctrl->status != 0) return;
  if (pred == 2 && ctrl->pcg_status != 0) return;
  __shared__ double sh[33];
  const int row0 = blockIdx.x * R;
  double acc[R];
#pragma unroll
  for (int r = 0; r < R; r++) acc[r] = 0.0;
  const int64_t n2 = ncols >> 1;
  // 4 independent 128-bit loads per row in flight per thread
  for (int64_t j = threadIdx.x; j < n2; j += 256 * 4) {
    double2 vv[4];
#pragma unroll
    for (int u = 0; u < 4; u++) {
      int64_t jj = j + (int64_t)u * 256;
      vv[u] = (jj < n2) ? *reinterpret_cast<const double2 *>(v + 2 * jj) : make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
      if (row0 + r < m) {
        const double *row = J + (int64_t)(row0 + r) * ld;
        const unsigned char *nzr = SKIP ? nz + (int64_t)((row0 + r) >> 6) * nz_ld : nullptr;
        double2 a[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          int64_t jj = j + (int64_t)u * 256;
          a[u] = (jj < n2 && (!SKIP || nzr[jj >> 3])) ? ld_stream2(row + 2 * jj) : make_double2(0.0, 0.0);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) acc[r] += a[u].x * vv[u].x + a[u].y * vv[u].y;
      }
    }
  }
  if ((ncols & 1) && threadIdx.x == 0) {
#pragma unroll
    for (int r = 0; r < R; r++) if (row0 + r < m) acc[r] += J[(int64_t)(row0 + r) * ld + ncols - 1] * v[ncols - 1];
  }
#pragma unroll
  for (int r = 0; r < R; r++) {
    double s = block_sum(acc[r], sh);
    if (threadIdx.x == 0 && row0 + r < m) t[row0 + r] = s;
  }
}

// ------------------------------------------------------------------ pass 2: cpart[rs][j] = sum_{i in split rs} J[i][j] u[i]
// CTA = 512 columns (2 per thread) x one row split; u chunk staged in shared memory.
template <bool SKIP = false>
__global__ void __launch_bounds__(256) cols_dot_kernel(const double *__restrict__ J, int64_t ld, int m, int64_t ncols,
                                                       const double *__restrict__ u, double *__restrict__ cpart,
                                                       int rows_per_split, const LargeCtrl *ctrl, int pred,
                                                       const unsigned char *__restrict__ nz = nullptr, int64_t nz_ld = 0) {
  if (pred == 1 && ctrl->status != 0) return;
  if (pred == 2 && ctrl->pcg_status != 0) return;
  extern __shared__ double us[];
  const int rs = blockIdx.y;
  const int i0 = rs * rows_per_split, i1 = min(m, i0 + rows_per_split);
  for (int i = threadIdx.x; i < i1 - i0; i += 256) us[i] = u[i0 + i];
  __syncthreads();
  const int64_t c = ((int64_t)blockIdx.x * 256 + threadIdx.x) * 2;
  if (c >= ncols) return;
  const bool pair = (c + 1 < ncols);
  double a0 = 0.0, a1 = 0.0;
  const double *base = J + (int64_t)i0 * ld + c;
  int i = 0;
  const int nr = i1 - i0;
  const unsigned char *nzc = SKIP ? nz + (c >> 4) : nullptr;   // this thread's K chunk; one map row per 64 rows of J
  if (pair) {
    for (; i + 8 <= nr; i += 8) {
      if (SKIP && !(nzc[(int64_t)((i0 + i) >> 6) * nz_ld] | nzc[(int64_t)((i0 + i + 7) >> 6) * nz_ld])) continue;   // 8 zero rows: a += 0 * w
      double2 q[8];
#pragma unroll
      for (int k = 0; k < 8; k++) q[k] = ld_stream2(base + (int64_t)(i + k) * ld);
#pragma unroll
      for (int k = 0; k < 8; k++) { double w = us[i + k]; a0 += q[k].x * w; a1 += q[k].y * w; }
    }
    for (; i < nr; i++) {
      if (SKIP && !nzc[(int64_t)((i0 + i) >> 6) * nz_ld]) continue;
      double2 q = ld_stream2(base + (int64_t)i * ld); double w = us[i]; a0 += q.x * w; a1 += q.y * w;
    }
    double *dst = cpart + (int64_t)rs * ncols + c;
    if (ncols & 1) { dst[0] = a0; dst[1] = a1; }   // odd row pitch: the rows of splits rs >= 1 start at odd offsets
    else *reinterpret_cast<double2 *>(dst) = make_double2(a0, a1);
  } else {
    for (; i < nr; i++) a0 += base[(int64_t)i * ld] * us[i];
    cpart[(int64_t)rs * ncols + c] = a0;
  }
}
// entry j of J'u from the row splits a column pass left in cpart (row pitch ld): s + cpart[0][j] + cpart[1][j] + ..., in that order
__device__ __forceinline__ double split_sum(const double *cpart, int nsplit, int64_t ld, int64_t j, double s = 0.0) {
  for (int k = 0; k < nsplit; k++) s += cpart[(int64_t)k * ld + j];
  return s;
}

// ------------------------------------------------------------------ triangular GEMVs: out[i] = sum_k T[i][k] in[k]
// lower: k <= i ; upper: k >= i.  One warp per row; `in` staged in shared memory.
// bf (optional, nblk <= 64): block structure of L^-1 (large_gemm.cuh::block_nz_kernel on Linv; XT = Linv' uses the transposed
// entry): terms of structurally zero 64 x 64 blocks are not loaded -- same lanes, same order, only "+ 0 * in[k]" terms less.
__global__ void __launch_bounds__(256) tri_gemv_kernel(const double *__restrict__ T, int64_t ld, int m,
                                                       const double *__restrict__ in, double *__restrict__ out, int upper,
                                                       double *__restrict__ out2, const LargeCtrl *ctrl, int pred,
                                                       const int *__restrict__ bf = nullptr, int nblk = 0) {
  if (pred == 1 && ctrl->status != 0) return;
  if (pred == 2 && ctrl->pcg_status != 0) return;
  extern __shared__ double ins[];
  for (int i = threadIdx.x; i < m; i += 256) ins[i] = in[i];
  __syncthreads();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (row >= m) return;
  const int k0 = upper ? row : 0, k1 = upper ? m : row + 1;
  const double *tr = T + (int64_t)row * ld;
  double s = 0.0;
  if (bf) {
    const int ib = row >> 6;
    unsigned long long mask = 0ULL;   // bit jb: block (ib, jb) of this triangle may be non-zero
    {
      const int j0 = lane, j1 = lane + 32;
      const int f0 = (j0 < nblk) ? (upper ? bf[(int64_t)j0 * nblk + ib] : bf[(int64_t)ib * nblk + j0]) : 0;
      const int f1 = (j1 < nblk) ? (upper ? bf[(int64_t)j1 * nblk + ib] : bf[(int64_t)ib * nblk + j1]) : 0;
      mask = (unsigned long long)__ballot_sync(0xffffffffu, f0 != 0) | ((unsigned long long)__ballot_sync(0xffffffffu, f1 != 0) << 32);
    }
    for (int k = k0 + lane; k < k1; k += 32) if ((mask >> (k >> 6)) & 1ULL) s += tr[k] * ins[k];
  } else
  for (int k = k0 + lane; k < k1; k += 32) s += tr[k] * ins[k];
  s = warp_sum(s);
  if (lane == 0) { out[row] = s; if (out2) out2[row] = s; }
}

// ------------------------------------------------------------------ finalize: ctrl->s[k] = reduce(part[slot k]) for the slots in mask
// bit k of summask: sum-reduce slot k into s[k]; bit k of maxmask: max-reduce slot k into s[k]
// explicit-inverse guard of the fused projcg (large.cu::factorize): an UPPER bound of cond(G) from quantities that are
// cheap once G^-1 is explicit: trace(G) = |L|_F^2 >= lambda_max(G), and lambda_max(G^-1) = 1 / lambda_min(G) by a few
// power iterations on G^-1 (each one m x m matvec).
__global__ void __launch_bounds__(256) lower_fro2_kernel(const double *__restrict__ L, int64_t ld, int m, double *part) {
  __shared__ double sh[33];
  double s = 0.0;
  for (int i = blockIdx.x; i < m; i += gridDim.x) {
    const double *row = L + (int64_t)i * ld;
    for (int k = threadIdx.x; k <= i; k += blockDim.x) s += row[k] * row[k];
  }
  s = block_sum(s, sh);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}
// v <- w / |w| ; ctrl->ldiag_min = 1 / |w| (the running estimate of lambda_min(G)); first call (w == nullptr): v = 1/sqrt(m)
// and ctrl->ldiag_max = sum(part) = trace(G)
__global__ void __launch_bounds__(256) power_step_kernel(int m, const double *w, double *v, const double *part, int np, LargeCtrl *ctrl) {
  __shared__ double sh[33];
  if (!w) {
    const double tr = reduce_partials(part, np, sh);
    for (int i = threadIdx.x; i < m; i += blockDim.x) v[i] = rsqrt((double)m);
    if (threadIdx.x == 0) { ctrl->ldiag_max = tr; ctrl->ldiag_min = 0.0; }
    return;
  }
  double s = 0.0;
  for (int i = threadIdx.x; i < m; i += blockDim.x) s += w[i] * w[i];
  s = sqrt(block_sum(s, sh));
  for (int i = threadIdx.x; i < m; i += blockDim.x) v[i] = w[i] / s;
  if (threadIdx.x == 0) ctrl->ldiag_min = 1.0 / s;
}

__global__ void __launch_bounds__(256) finalize_kernel(const double *part, int np, unsigned summask, unsigned maxmask,
                                                       LargeCtrl *ctrl) {
  __shared__ double sh[33];
  for (int k = 0; k < NSLOT; k++) {
    if (summask & (1u << k)) { double r = reduce_partials(part + (size_t)k * MAXP, np, sh); if (threadIdx.x == 0) ctrl->s[k] = r; }
    else if (maxmask & (1u << k)) { double r = reduce_partials_max(part + (size_t)k * MAXP, np, sh); if (threadIdx.x == 0) ctrl->s[k] = r; }
    __syncthreads();
  }
}

// part[0] = sum of the first `used` partials of slot 0, part[1..np) = 0  (single CTA, fixed order)
__global__ void __launch_bounds__(256) collapse_partials_kernel(double *part, int used, int np) {
  __shared__ double sh[33];
  double r = reduce_partials(part, used, sh);
  __syncthreads();
  for (int i = threadIdx.x; i < max(np, used); i += 256) part[i] = (i == 0) ? r : 0.0;
}

// ------------------------------------------------------------------ generic fused elementwise kernel with up to 3 sum partials + 1 max
// f(i, acc): elementwise body for index i; acc[0..2] are sum-reduced into slots s0..s0+2, acc[3] max-reduced into slot s0+3
template <class F>
__global__ void __launch_bounds__(256) vec_kernel(int64_t n, F f, double *part, int s0, int nsum, int domax) {
  __shared__ double sh[33];
  double acc[4] = {0.0, 0.0, 0.0, 0.0};
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) f(i, acc);
  for (int k = 0; k < nsum; k++) {
    double r = block_sum(acc[k], sh);
    if (threadIdx.x == 0) part[(size_t)(s0 + k) * MAXP + blockIdx.x] = r;
  }
  if (domax) {
    double r = block_max(acc[3], sh);
    if (threadIdx.x == 0) part[(size_t)(s0 + 3) * MAXP + blockIdx.x] = r;
  }
}

// ------------------------------------------------------------------ projcg! iteration pieces (projcg.jl:71-112)
// Loop partial slots (buffer `lp`): 0 = d.Ad (written by the family's hess kernel), 1 = rp.gp, 2+par = gp.gp of the
// iteration with parity par.  rg of iteration k is gp.gp of iteration k-1 (r == g after every projection), so it is
// re-reduced from slot 2+(par^1) instead of being stored: no CTA ever reads a scalar that another CTA of the same
// grid writes, and no grid-wide sync or extra "flip" launch is needed.  `par` = k & 1 comes from the host.
// Status writes by CTA 0 are benign races: every CTA derives the same decision from the same partials.
//
// update1: alpha = rg/dAd ; x += alpha d ; rp = r + alpha Ad      (negative-curvature / rg<=0 exits decided here)
__global__ void __launch_bounds__(256) cg_update1_kernel(int64_t n, double *__restrict__ xs, const double *__restrict__ d,
                                                         const double *__restrict__ r, const double *__restrict__ Ad,
                                                         double *__restrict__ rp, const double *lp, int np_hess, int np_vec,
                                                         int par, LargeCtrl *ctrl) {
  if (ctrl->status != 0) return;
  __shared__ double sh[33];
  const double dAd = reduce_partials(lp + 0 * MAXP, np_hess, sh);
  const double rg = reduce_partials(lp + (2 + (par ^ 1)) * MAXP, np_vec, sh);
  int st = 0;
  if (dAd <= 0.0) st = 2;            // projcg.jl:77-82
  else if (rg <= 0.0) st = 3;        // :87-89
  const double alpha = rg / dAd;
  if (st == 0) {
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
      xs[i] += alpha * d[i];
      rp[i] = r[i] + alpha * Ad[i];
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    ctrl->dAd = dAd; ctrl->alpha = alpha; ctrl->rg = rg; ctrl->iter = ctrl->iter + 1;
    if (st != 0) ctrl->status = st;
  }
}
// update2: gp = rp - sum_rs cpart[rs] ; partials rp.gp (slot 1), gp.gp (slot 2+par)
__global__ void __launch_bounds__(256) cg_update2_kernel(int64_t n, const double *__restrict__ rp, double *__restrict__ gp,
                                                         const double *__restrict__ cpart, int nsplit, double *lp, int par,
                                                         const LargeCtrl *ctrl, int pred) {
  if (pred && ctrl->status != 0) return;
  __shared__ double sh[33];
  double a = 0.0, b = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const double s = split_sum(cpart, nsplit, n, i);
    double rpi = rp[i], g = rpi - s;
    gp[i] = g; a += rpi * g; b += g * g;
  }
  a = block_sum(a, sh); b = block_sum(b, sh);
  if (threadIdx.x == 0) { lp[1 * MAXP + blockIdx.x] = a; lp[(2 + par) * MAXP + blockIdx.x] = b; }
}
// update3: beta = rp.gp/rg ; d = beta d - gp ; r = gp ; nr = |gp| ; convergence / limit tests (projcg.jl:98-111)
__global__ void __launch_bounds__(256) cg_update3_kernel(int64_t n, double *__restrict__ d, double *__restrict__ r,
                                                         const double *__restrict__ gp, const double *lp, int np, int par,
                                                         LargeCtrl *ctrl) {
  if (ctrl->status != 0) return;
  __shared__ double sh[33];
  const double rpgp = reduce_partials(lp + 1 * MAXP, np, sh);
  const double gg = reduce_partials(lp + (2 + par) * MAXP, np, sh);
  const double rg = reduce_partials(lp + (2 + (par ^ 1)) * MAXP, np, sh);
  const double beta = rpgp / rg;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    double g = gp[i];
    d[i] = beta * d[i] - g; r[i] = g;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    const double nr = sqrt(gg);
    ctrl->beta = beta; ctrl->rpgp = rpgp; ctrl->gg = gg; ctrl->nr = nr;
    if (nr < ctrl->tol) ctrl->status = 1; else if (ctrl->iter >= ctrl->lim) ctrl->status = 4;
  }
}

// after the start-up projection of projcg! (projcg.jl:58-62): r = g = r - sum cpart ; d = -g ; r.r partials -> slot 3
__global__ void __launch_bounds__(256) cg_init_kernel(int64_t n, double *__restrict__ r, double *__restrict__ d,
                                                      const double *__restrict__ cpart, int nsplit, double *lp) {
  __shared__ double sh[33];
  double a = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const double s = split_sum(cpart, nsplit, n, i);
    double g = r[i] - s;
    r[i] = g; d[i] = -1.0 * g; a += g * g;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[3 * MAXP + blockIdx.x] = a;
}
// Hessian action of a family whose Lagrangian Hessian is diagonal (DIAGQUAD): dest = hdiag .* src, partial src.dest -> slot 0
__global__ void __launch_bounds__(256) hess_diag_kernel(int64_t n, const double *__restrict__ hd, const double *__restrict__ src,
                                                        double *__restrict__ dest, double *lp, const LargeCtrl *ctrl, int pred) {
  if (pred == 1 && ctrl->status != 0) return;
  __shared__ double sh[33];
  double a = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    double v = src[i], h = hd[i] * v;
    dest[i] = h; a += v * h;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[0 * MAXP + blockIdx.x] = a;
}
// ProjPenalty right-hand side (retractions.jl:369-371 + pcg!'s fill!(p,0)): g = sum cpart + mu g ; dx = 0 ; r = g ; p = 0 ;
// r.r partials -> slot 5 (rho of pcg iteration 0)
__global__ void __launch_bounds__(256) pp_rhs_kernel(int64_t n, double *__restrict__ g, double *__restrict__ dx,
                                                     double *__restrict__ r, double *__restrict__ p,
                                                     const double *__restrict__ cpart, int nsplit, double mu, double *lp) {
  __shared__ double sh[33];
  double a = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    double gi = split_sum(cpart, nsplit, n, i) + mu * g[i];
    g[i] = gi; dx[i] = 0.0; r[i] = gi; p[i] = 0.0; a += gi * gi;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[5 * MAXP + blockIdx.x] = a;
}

// pcg! start state for the unit-level export: x = 0, p = 0, r.r partials -> slot 5
__global__ void __launch_bounds__(256) pcg_start_kernel(int64_t n, const double *__restrict__ r, double *__restrict__ dx,
                                                        double *__restrict__ p, double *lp) {
  __shared__ double sh[33];
  double a = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    dx[i] = 0.0; p[i] = 0.0; double ri = r[i]; a += ri * ri;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[5 * MAXP + blockIdx.x] = a;
}

// ------------------------------------------------------------------ pcg! iteration pieces (retractions.jl:207-238), M! = copy
// Loop partial slots: 4 = p.z, 5+par = r.r at the START of the iteration with parity par (rho_k); rho_{k-1} is still
// in slot 5+(par^1) when pcg_a(k) runs.  first = 1 for k = 0 (rho_prev = 1, norm_res = Inf: retractions.jl:202-203).
__global__ void __launch_bounds__(256) pcg_a_kernel(int64_t n, double *__restrict__ p, const double *__restrict__ r,
                                                    const double *lp, int np, int par, int first, LargeCtrl *ctrl) {
  if (ctrl->pcg_status != 0) return;
  __shared__ double sh[33];
  const double rho = reduce_partials(lp + (5 + par) * MAXP, np, sh);
  const double rho_prev = first ? 1.0 : reduce_partials(lp + (5 + (par ^ 1)) * MAXP, np, sh);
  const double norm_res = first ? INFINITY : sqrt(rho);
  int st = 0;
  if (!(norm_res > ctrl->tol)) st = 1; else if (ctrl->pcg_iter >= ctrl->pcg_lim) st = 4;
  const double beta = rho / rho_prev;
  if (st == 0) {
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) p[i] = r[i] + beta * p[i];
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) { ctrl->norm_res = norm_res; ctrl->rho = rho; if (st != 0) ctrl->pcg_status = st; }
}
// z = sum_rs cpart + mu p ; partial p.z (slot 4)
__global__ void __launch_bounds__(256) pcg_z_kernel(int64_t n, double *__restrict__ z, const double *__restrict__ p,
                                                    const double *__restrict__ cpart, int nsplit, double *lp,
                                                    const LargeCtrl *ctrl) {
  if (ctrl->pcg_status != 0) return;
  __shared__ double sh[33];
  const double mu = ctrl->mu;
  double a = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    const double s = split_sum(cpart, nsplit, n, i);
    double pi = p[i], zi = s + mu * pi;
    z[i] = zi; a += pi * zi;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[4 * MAXP + blockIdx.x] = a;
}
// alpha = rho / p.z ; x += alpha p ; r -= alpha z ; partial r.r -> slot 5+(par^1) (rho of the next iteration)
__global__ void __launch_bounds__(256) pcg_x_kernel(int64_t n, double *__restrict__ x, double *__restrict__ r,
                                                    const double *__restrict__ p, const double *__restrict__ z, double *lp,
                                                    int np, int par, LargeCtrl *ctrl) {
  if (ctrl->pcg_status != 0) return;
  __shared__ double sh[33];
  const double pz = reduce_partials(lp + 4 * MAXP, np, sh);
  const double rho = reduce_partials(lp + (5 + par) * MAXP, np, sh);
  const double alpha = rho / pz;
  double a = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) {
    x[i] += alpha * p[i];
    double ri = r[i] - alpha * z[i];
    r[i] = ri; a += ri * ri;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[(5 + (par ^ 1)) * MAXP + blockIdx.x] = a;
  if (blockIdx.x == 0 && threadIdx.x == 0) { ctrl->pz = pz; ctrl->alpha = alpha; ctrl->pcg_iter = ctrl->pcg_iter + 1; }
}

}  // namespace lfpsqp
