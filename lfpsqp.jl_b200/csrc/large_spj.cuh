// large_spj.cuh -- LFPSQP_FAM_SPARSE_QCQP_CSR: the Jacobian of the sparse QCQP family kept sparse on the device.
//
// J is stored twice, by value: in CSR order (row pointers = the constraint pointers con_ptr, column indices = the segment rows
// seg_row of large_spq.cu) and in CSC order (SpjDev::cptr / crow).  Every kernel sums in an order fixed by the sparsity pattern
// alone (never by the SM count or the grid size) and without floating-point atomics, so two solves are bit-identical.
//
//   spj_cjac  jac!   c(x) and the structural entries of J, written once into each value array
//   spj_rows  t = J v         one warp per row; a row longer than SPJ_CHUNK entries is cut into pattern-fixed chunks (slots)
//                             whose partial sums spj_combine adds in chunk order
//   spj_cols  y = J' u        one thread per column, rows in increasing order
//   spj_gram  G = J W J'      lower triangle, W = I or diag(Dy^2); one warp per row i of G scatters into a shared m-vector:
//                             for each entry (i, j) in column order, the entries (k <= i, j) of column j are distinct in k and
//                             are added in parallel.  Work: sum_j nnz(col j)^2, no m n term.  Long rows: partial rows per
//                             chunk, summed in chunk order by spj_gram_combine.
// Predication (pred 0 / 1 / 2 tested against ctrl->status / pcg_status) as rows_dot_kernel.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "large_ctrl.h"
#include "large_device.cuh"

namespace lfpsqp {

__device__ __forceinline__ bool spj_skip(const LargeCtrl *ctrl, int pred) {
  return (pred == 1 && ctrl->status != 0) || (pred == 2 && ctrl->pcg_status != 0);
}
// work item of the row-shaped kernels: items [0, m) are rows (a long row's item does nothing), items [m, m + nslot) chunks
// of long rows.  -> [b, e) segment range, or false when the item has nothing to do
__device__ __forceinline__ bool spj_item(const SpjDev &P, const int *__restrict__ con_ptr, int64_t item, int &b, int &e) {
  if (item < P.m) {
    const int i = (int)item;
    if (P.row_slot[i + 1] > P.row_slot[i]) return false;
    b = con_ptr[i]; e = con_ptr[i + 1];
    return true;
  }
  const int64_t s = item - P.m;
  if (s >= P.nslot) return false;
  b = P.slot_beg[s]; e = P.slot_end[s];
  return true;
}

// jac!: one warp per item.  cval[i] = sum over the segments (i, r) of x_r (1/2 (Qc_i x)_r + Ac[i, r]) - bc[i] (chunk partials
// of a long row -> part[slot]); with WRITE_J also J[i, r] = (Qc_i x)_r + Ac[i, r] into jr (CSR order) and jc (CSC order)
template <bool WRITE_J>
__global__ void __launch_bounds__(256) spj_cjac_kernel(SpjDev P, const int *__restrict__ con_ptr, const int *__restrict__ seg_row,
                                                       const double *__restrict__ seg_a, const int *__restrict__ seg_ptr,
                                                       const int *__restrict__ seg_col, const double *__restrict__ seg_val,
                                                       const double *__restrict__ bc, const double *__restrict__ x,
                                                       double *__restrict__ cval, double *__restrict__ part) {
  const int64_t item = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  int b, e;
  if (!spj_item(P, con_ptr, item, b, e)) return;
  double acc = 0.0;
  for (int s = b + lane; s < e; s += 32) {
    double qx = 0.0;
    for (int k = seg_ptr[s]; k < seg_ptr[s + 1]; k++) qx += seg_val[k] * x[seg_col[k]];
    const int r = seg_row[s];
    const double a = seg_a[s];
    acc += x[r] * (0.5 * qx + a);
    if (WRITE_J) { const double v = qx + a; P.jr[s] = v; P.jc[P.csc_of[s]] = v; }
  }
  acc = warp_sum(acc);
  if (lane == 0) {
    if (item < P.m) cval[item] = acc - bc[item];
    else part[item - P.m] = acc;
  }
}

// t = J v over CSR: one warp per item (short row -> t[i], chunk of a long row -> part[slot])
__global__ void __launch_bounds__(256) spj_rows_kernel(SpjDev P, const int *__restrict__ con_ptr, const int *__restrict__ col,
                                                       const double *__restrict__ v, double *__restrict__ t, double *__restrict__ part,
                                                       const LargeCtrl *ctrl, int pred) {
  if (spj_skip(ctrl, pred)) return;
  const int64_t item = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  int b, e;
  if (!spj_item(P, con_ptr, item, b, e)) return;
  double acc = 0.0;
  for (int s = b + lane; s < e; s += 32) acc += P.jr[s] * v[col[s]];
  acc = warp_sum(acc);
  if (lane == 0) {
    if (item < P.m) t[item] = acc;
    else part[item - P.m] = acc;
  }
}

// out[i] = sum of the chunk partials of long row i in chunk order (- b[i] when b is given): one thread per long row
__global__ void __launch_bounds__(256) spj_combine_kernel(SpjDev P, const double *__restrict__ part, const double *__restrict__ b,
                                                          double *__restrict__ out, const LargeCtrl *ctrl, int pred) {
  if (spj_skip(ctrl, pred)) return;
  const int r = blockIdx.x * 256 + threadIdx.x;
  if (r >= P.nlong) return;
  const int i = P.long_row[r];
  double s = 0.0;
  for (int q = P.row_slot[i]; q < P.row_slot[i + 1]; q++) s += part[q];
  out[i] = b ? s - b[i] : s;
}

// y = J' u over CSC: one thread per column, rows in increasing order
__global__ void __launch_bounds__(256) spj_cols_kernel(SpjDev P, int64_t n, const double *__restrict__ u, double *__restrict__ y,
                                                       const LargeCtrl *ctrl, int pred) {
  if (spj_skip(ctrl, pred)) return;
  for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < n; j += (int64_t)gridDim.x * 256) {
    double s = 0.0;
    const int p1 = P.cptr[j + 1];
    for (int p = P.cptr[j]; p < p1; p++) s += P.jc[p] * u[P.crow[p]];
    y[j] = s;
  }
}

// G[i][k] (k <= i) = sum_j (J_ij w_j) (J_kj w_j), w = Dy (WEIGHTED) or 1.  One warp per item; the shared m-vector acc holds row i.
// Columns are visited in CSR order; the column data of 32 consecutive entries is fetched by the 32 lanes at once and
// broadcast.  Within one column the rows k are distinct, so the lanes add in parallel; __syncwarp orders the columns.
template <bool WEIGHTED>
__global__ void __launch_bounds__(32) spj_gram_kernel(SpjDev P, const int *__restrict__ con_ptr, const int *__restrict__ col,
                                                      const double *__restrict__ w, double *__restrict__ G, int64_t ldm,
                                                      double *__restrict__ gpart) {
  extern __shared__ double acc[];
  const int64_t item = blockIdx.x;
  const int lane = threadIdx.x;
  int b, e;
  if (!spj_item(P, con_ptr, item, b, e)) return;
  const int i = (item < P.m) ? (int)item : P.slot_row[item - P.m];
  for (int k = lane; k <= i; k += 32) acc[k] = 0.0;
  __syncwarp();
  for (int s0 = b; s0 < e; s0 += 32) {
    const int s = s0 + lane;
    int p0 = 0, p1 = 0;
    double a = 0.0, wj = 1.0;
    if (s < e) {
      const int j = col[s];
      if (WEIGHTED) wj = w[j];
      a = P.jr[s] * wj;
      p0 = P.cptr[j]; p1 = P.cptr[j + 1];
    }
    const int cnt = min(32, e - s0);
    for (int q = 0; q < cnt; q++) {
      const int q0 = __shfl_sync(0xffffffffu, p0, q), q1 = __shfl_sync(0xffffffffu, p1, q);
      const double qa = __shfl_sync(0xffffffffu, a, q), qw = WEIGHTED ? __shfl_sync(0xffffffffu, wj, q) : 1.0;
      for (int p = q0 + lane; p < q1; p += 32) {
        const int k = P.crow[p];
        if (k > i) break;   // rows of a column are increasing: the rest is above the diagonal
        acc[k] += qa * (WEIGHTED ? P.jc[p] * qw : P.jc[p]);
      }
      __syncwarp();
    }
  }
  double *dst = (item < P.m) ? G + (int64_t)i * ldm : gpart + (item - P.m) * (int64_t)P.m;
  for (int k = lane; k <= i; k += 32) dst[k] = acc[k];
}

// G[i][k] (k <= i) of long row i = sum of its chunks' partial rows in chunk order; grid (k blocks, long rows)
__global__ void __launch_bounds__(256) spj_gram_combine_kernel(SpjDev P, const double *__restrict__ gpart, double *__restrict__ G,
                                                               int64_t ldm) {
  const int i = P.long_row[blockIdx.y];
  const int k = blockIdx.x * 256 + threadIdx.x;
  if (k > i) return;
  double s = 0.0;
  for (int q = P.row_slot[i]; q < P.row_slot[i + 1]; q++) s += gpart[(int64_t)q * P.m + k];
  G[(int64_t)i * ldm + k] = s;
}

}  // namespace lfpsqp
