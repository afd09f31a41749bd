// large_families.cuh -- device callbacks of the benchmark families for the large-n mode (whole-GPU kernels).
// Same contract as the batched callbacks (src/autodiff_generators.jl:7-9, :40-42, :80-104), but every call is a
// grid-wide kernel over the column shard [col0, col0+n_loc) this GPU owns.
#pragma once
#include "large_kernels.cuh"

namespace lfpsqp {

// ================================================================== DIAGQUAD (BASELINE config C5)
// c_i = 1/2 sum_j Q_ij x_j^2 + A_i.x - b_i ; f = 1/2 sum_j w_j (x_j - xt_j)^2 ; Q, A: m x n_loc row-major shards.

// raw row sums s_i = sum_j (1/2 Q_ij x_j + A_ij) x_j  (b is subtracted after the cross-GPU reduction);
// WRITE_J also stores J_ij = Q_ij x_j + A_ij (jac!, which "also writes cval": autodiff_generators.jl:40-42)
template <int R, bool WRITE_J>
__global__ void __launch_bounds__(256) dq_rows_kernel(const double *__restrict__ Q, const double *__restrict__ A, int64_t ld,
                                                      int m, int64_t ncols, const double *__restrict__ x,
                                                      double *__restrict__ J, double *__restrict__ rows) {
  __shared__ double sh[33];
  const int row0 = blockIdx.x * R;
  double acc[R];
#pragma unroll
  for (int r = 0; r < R; r++) acc[r] = 0.0;
  const int64_t n2 = ncols >> 1;
  for (int64_t j = threadIdx.x; j < n2; j += 256 * 2) {
    double2 xv[2];
#pragma unroll
    for (int u = 0; u < 2; u++) {
      int64_t jj = j + (int64_t)u * 256;
      xv[u] = (jj < n2) ? *reinterpret_cast<const double2 *>(x + 2 * jj) : make_double2(0.0, 0.0);
    }
#pragma unroll
    for (int r = 0; r < R; r++) {
      if (row0 + r >= m) continue;
      const int64_t off = (int64_t)(row0 + r) * ld;
      double2 q[2], a[2];
#pragma unroll
      for (int u = 0; u < 2; u++) {
        int64_t jj = j + (int64_t)u * 256;
        q[u] = (jj < n2) ? ld_stream2(Q + off + 2 * jj) : make_double2(0.0, 0.0);
        a[u] = (jj < n2) ? ld_stream2(A + off + 2 * jj) : make_double2(0.0, 0.0);
      }
#pragma unroll
      for (int u = 0; u < 2; u++) {
        int64_t jj = j + (int64_t)u * 256;
        acc[r] += (0.5 * q[u].x * xv[u].x + a[u].x) * xv[u].x + (0.5 * q[u].y * xv[u].y + a[u].y) * xv[u].y;
        if (WRITE_J && jj < n2)
          *reinterpret_cast<double2 *>(J + off + 2 * jj) = make_double2(q[u].x * xv[u].x + a[u].x, q[u].y * xv[u].y + a[u].y);
      }
    }
  }
  if ((ncols & 1) && threadIdx.x == 0) {
    int64_t jl = ncols - 1;
#pragma unroll
    for (int r = 0; r < R; r++) if (row0 + r < m) {
      int64_t off = (int64_t)(row0 + r) * ld + jl;
      acc[r] += (0.5 * Q[off] * x[jl] + A[off]) * x[jl];
      if (WRITE_J) J[off] = Q[off] * x[jl] + A[off];
    }
  }
#pragma unroll
  for (int r = 0; r < R; r++) {
    double s = block_sum(acc[r], sh);
    if (threadIdx.x == 0 && row0 + r < m) rows[row0 + r] = s;
  }
}

// ================================================================== THOMSON (BASELINE config C4)
// Pairwise O(N^2) kernels on a 2-D grid: blockIdx.x = block of 256 OWNED points i, blockIdx.y = chunk of the j range (so
// that N = 4096 fills the GPU: 16 x 16 CTAs instead of 16).  Points j are staged through shared memory.
// Column-sharded (SURVEY.md 8e-iv): this rank owns the points [i0, i0 + npl) (their 3 npl coordinates are its columns of J
// and its entries of every n-vector); x / v are the ALL-GATHERED coordinates of all np_ points, outputs are local.
// mode 0: f partials (sum_{j!=i} 1/r_ij, halved)                       -> part slot s0 [blockIdx.y * gridDim.x + blockIdx.x]
// mode 1: partial gradient   -sum_j (x_i-x_j)/r^3                      -> ws[blockIdx.y][3 i ..]
// mode 2: partial Hessian action sum_j [3 r (r.w)/r^5 - w/r^3], w = v_i - v_j  -> ws[blockIdx.y][3 i ..]
template <int MODE>
__global__ void __launch_bounds__(256) thomson_pair_kernel(int np_, int i0, int npl, const double *__restrict__ x, const double *__restrict__ v,
                                                           double *__restrict__ ws, double *part, int s0,
                                                           const LargeCtrl *ctrl, int pred) {
  if (pred == 1 && ctrl->status != 0) return;
  __shared__ double xs[256 * 3];
  __shared__ double vs[MODE == 2 ? 256 * 3 : 3];
  __shared__ double sh[33];
  const int il = blockIdx.x * 256 + threadIdx.x;      // local index of the owned point
  const int i = i0 + il;
  const bool act = il < npl;
  const int jlen = (np_ + gridDim.y - 1) / gridDim.y, jbeg = blockIdx.y * jlen, jend = min(np_, jbeg + jlen);
  double xi = 0, yi = 0, zi = 0, vx = 0, vy = 0, vz = 0;
  if (act) { xi = x[3 * i]; yi = x[3 * i + 1]; zi = x[3 * i + 2]; if (MODE == 2) { vx = v[3 * i]; vy = v[3 * i + 1]; vz = v[3 * i + 2]; } }
  double a0 = 0, a1 = 0, a2 = 0;
  for (int j0 = jbeg; j0 < jend; j0 += 256) {
    __syncthreads();
    int jn = min(256, jend - j0);
    for (int e = threadIdx.x; e < jn * 3; e += 256) { xs[e] = x[3 * j0 + e]; if (MODE == 2) vs[e] = v[3 * j0 + e]; }
    __syncthreads();
    if (act) {
      for (int jj = 0; jj < jn; jj++) {
        if (j0 + jj == i) continue;
        double a = xi - xs[3 * jj], b = yi - xs[3 * jj + 1], c = zi - xs[3 * jj + 2];
        double r2 = a * a + b * b + c * c;
        if (MODE == 0) { a0 += 1.0 / sqrt(r2); }
        else if (MODE == 1) { double ir3 = 1.0 / (r2 * sqrt(r2)); a0 -= a * ir3; a1 -= b * ir3; a2 -= c * ir3; }
        else {
          double wa = vx - vs[3 * jj], wb = vy - vs[3 * jj + 1], wc = vz - vs[3 * jj + 2];
          double ir3 = 1.0 / (r2 * sqrt(r2)), ir5 = ir3 / r2, rw = 3.0 * (a * wa + b * wb + c * wc) * ir5;
          a0 += rw * a - wa * ir3; a1 += rw * b - wb * ir3; a2 += rw * c - wc * ir3;
        }
      }
    }
  }
  if (MODE == 0) {
    double pr = block_sum(act ? 0.5 * a0 : 0.0, sh);
    if (threadIdx.x == 0) part[(size_t)s0 * MAXP + blockIdx.y * gridDim.x + blockIdx.x] = pr;
  } else if (act) {
    double *o = ws + (size_t)blockIdx.y * 3 * npl + 3 * il;
    o[0] = a0; o[1] = a1; o[2] = a2;
  }
}
// sums the j-chunk partials; mode 2 adds the constraint part 2 lam_i v_i and writes the v.dest partial (loop slot 0)
template <int MODE>
__global__ void __launch_bounds__(256) thomson_reduce_kernel(int np_, int chunks, const double *__restrict__ ws,
                                                             const double *__restrict__ v, const double *__restrict__ lam,
                                                             double *__restrict__ out, double *part, int s0,
                                                             const LargeCtrl *ctrl, int pred) {
  if (pred == 1 && ctrl->status != 0) return;
  __shared__ double sh[33];
  const int e = blockIdx.x * 256 + threadIdx.x, n3 = 3 * np_;
  double pr = 0.0;
  if (e < n3) {
    double s = 0.0;
    for (int k = 0; k < chunks; k++) s += ws[(size_t)k * n3 + e];
    if (MODE == 2) { double ve = v[e]; s += 2.0 * lam[e / 3] * ve; pr = ve * s; }
    out[e] = s;
  }
  if (MODE == 2) {
    pr = block_sum(pr, sh);
    if (threadIdx.x == 0) part[(size_t)s0 * MAXP + blockIdx.x] = pr;
  }
}
// c_i = |x_i|^2 - 1 for the owned points (x = this rank's coordinates; cval rows of the other ranks are left untouched:
// zeroed by the caller and summed over the ranks) ; optionally the three structural non-zeros of row i0 + i of the
// (dense-treated) Jacobian shard
__global__ void thomson_c_kernel(int npl, int i0, const double *__restrict__ x, double *__restrict__ cval, double *J, int64_t ld) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= npl) return;
  double a = x[3 * i], b = x[3 * i + 1], c = x[3 * i + 2];
  cval[i0 + i] = a * a + b * b + c * c - 1.0;
  if (J) { double *r = J + (int64_t)(i0 + i) * ld + 3 * i; r[0] = 2.0 * a; r[1] = 2.0 * b; r[2] = 2.0 * c; }
}

// ================================================================== SPARSE_QCQP (LFPSQP_FAM_SPARSE_QCQP, one GPU)
// f = 1/2 x'P x + q.x + r ; c_i = 1/2 x'Qc_i x + Ac_i.x - bc_i.  Structures: SpqDev (large_ctrl.h).  Every sum has a fixed
// order (no atomics): two solves of one problem are bit-identical.

// CSR pass y = A x with G lanes per row (rows handed out warp-uniformly, so every lane of a warp takes the shuffles)
//   MODE 0: f partial sum_r x_r (1/2 (Ax)_r + q_r) -> part[blockIdx.x] (block 0 adds r0)
//   MODE 1: y = A x + q (grad)
//   MODE 2: y = A x (Hessian action), partial x.y -> part[blockIdx.x] unless part is NULL; predicated on ctrl->status
template <int G, int MODE>
__global__ void __launch_bounds__(256) spq_csr_kernel(int64_t n, const int *__restrict__ rp, const int *__restrict__ ci,
                                                      const double *__restrict__ v, const double *__restrict__ x,
                                                      const double *__restrict__ q, double r0, double *__restrict__ y,
                                                      double *part, const LargeCtrl *ctrl, int pred) {
  if (MODE == 2 && pred == 1 && ctrl->status != 0) return;
  __shared__ double sh[33];
  constexpr int RPW = 32 / G;   // rows per warp and step
  const int lane = threadIdx.x & 31, sub = lane % G;
  const int64_t warp = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5, nwarp = (int64_t)gridDim.x * 8;
  double acc = 0.0;
  for (int64_t row0 = warp * RPW; row0 < n; row0 += nwarp * RPW) {
    const int64_t row = row0 + lane / G;
    double s = 0.0;
    if (row < n) {
      const int k1 = rp[row + 1];
      for (int k = rp[row] + sub; k < k1; k += G) s += v[k] * x[ci[k]];
    }
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (sub == 0 && row < n) {
      if (MODE == 0) acc += x[row] * (0.5 * s + q[row]);
      else if (MODE == 1) y[row] = s + q[row];
      else { y[row] = s; acc += x[row] * s; }
    }
  }
  if (MODE == 0 || (MODE == 2 && part)) {
    const double t = block_sum(acc, sh);
    if (threadIdx.x == 0) part[blockIdx.x] = (MODE == 0 && blockIdx.x == 0) ? t + r0 : t;
  }
}

// values of H on its union pattern: hval[e] = sum over the sources of e, in their stored order, of (P entry | lam_i Qc_i entry)
__global__ void __launch_bounds__(256) spq_hess_assemble_kernel(int64_t nh, const int *__restrict__ sp, const int *__restrict__ con,
                                                                const double *__restrict__ val, const double *__restrict__ lam,
                                                                double *__restrict__ hval) {
  for (int64_t e = (int64_t)blockIdx.x * 256 + threadIdx.x; e < nh; e += (int64_t)gridDim.x * 256) {
    double s = 0.0;
    for (int k = sp[e]; k < sp[e + 1]; k++) { const int i = con[k]; s += (i < 0) ? val[k] : lam[i] * val[k]; }
    hval[e] = s;
  }
}

// one CTA per constraint i: cval[i] = sum over the segments (i, r) of x_r (1/2 (Qc_i x)_r + Ac[i, r]) - bc[i], and with
// WRITE_J the structural entries J[i, r] = (Qc_i x)_r + Ac[i, r] (every other entry of J stays zero)
template <bool WRITE_J>
__global__ void __launch_bounds__(256) spq_cjac_kernel(const int *__restrict__ con_ptr, const int *__restrict__ seg_row,
                                                       const double *__restrict__ seg_a, const int *__restrict__ seg_ptr,
                                                       const int *__restrict__ seg_col, const double *__restrict__ seg_val,
                                                       const double *__restrict__ bc, const double *__restrict__ x,
                                                       double *__restrict__ J, int64_t ld, double *__restrict__ cval) {
  __shared__ double sh[33];
  const int i = blockIdx.x;
  double acc = 0.0;
  for (int s = con_ptr[i] + threadIdx.x; s < con_ptr[i + 1]; s += 256) {
    double qx = 0.0;
    for (int k = seg_ptr[s]; k < seg_ptr[s + 1]; k++) qx += seg_val[k] * x[seg_col[k]];
    const int r = seg_row[s];
    const double a = seg_a[s];
    acc += x[r] * (0.5 * qx + a);
    if (WRITE_J) J[(int64_t)i * ld + r] = qx + a;
  }
  const double t = block_sum(acc, sh);
  if (threadIdx.x == 0) cval[i] = t - bc[i];
}

}  // namespace lfpsqp
