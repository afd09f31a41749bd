// large_ineq.cuh -- bound embedding (src/inequality_helper.jl) of the large-n mode.
//
// With finite bounds the driver works on the 2n-vector [x ; y] (optimize.jl:172-182): every working vector of this
// mode is then stored as [x-half (nx = n_loc entries) | y-half (nx entries)] on each rank.  The SVD-based operators of
// the reference have closed forms in the Gram/Cholesky setting (DESIGN.md section 2, SURVEY App. B):
//   Q Q' v          = D D' v + PJct G_w^-1 PJct' v ,  G_w = J diag(Dy^2) J'                 (inequality_helper.jl:161-212)
//     a = Dx v_x + Dy v_y ; PJct' v = J (Dy (Dy v_x - Dx v_y)) ; w = J' G_w^-1 PJct' v
//     v_x -= Dx a + Dy^2 w ; v_y -= Dy a - Dx Dy w
//   lambda_y        = -(Dx/S) w + a/S                                                       (:286-308)
//   bigA' v         = [S (Dx v_x + Dy v_y) ; J v_x]   ,  bigA [wh ; wc] = [J' wc + Dx S wh ; Dy S wh]      (:215-271)
//   Hessian         = [H v_x + 2 lambda_y q v_x ; 2 lambda_y s v_y]                          (:144-158)
// The kernels below are the loop pieces (device-predicated like their unbounded twins in large_kernels.cuh); the
// one-off elementwise operations (generate_initial_y!, calculate_h!, inequality_gradient!, y_retract!) are lambdas
// in large.cu built from the device functions here.
#pragma once
#include "large_kernels.cuh"

namespace lfpsqp {


// calculate_h! (inequality_helper.jl:112-122)
__device__ __forceinline__ double ineq_h(double q, double r, double s, double t, double x, double y) {
  const double dx = x - r, dy = y - r;
  return q * (dx * dx) + (1.0 - q * q) * x + s * (dy * dy) - (1.0 - s * s) * y - t;
}
// generate_initial_y! (:92-109)
__device__ __forceinline__ double ineq_y0(double q, double r, double s, double t, double x) {
  if (q == 0.0 && s == 0.0) return x;                                             // line
  if (q == 0.0) return sqrt(fmax(-(x - t) / s, 0.0)) + r;                         // parabola
  return sqrt(fmax(t - (x - r) * (x - r), 0.0)) + r;                              // circle
}
// inequality_gradient! (:125-141): normalised (Dx, Dy) and the norm S
__device__ __forceinline__ void ineq_grad(double q, double r, double s, double x, double y, double &Dx, double &Dy, double &S) {
  const double dx = 2.0 * q * (x - r) + (q == 0.0 ? 1.0 : 0.0);
  const double dy = 2.0 * s * (y - r) - (s == 0.0 ? 1.0 : 0.0);
  const double sv = sqrt(dx * dx + dy * dy);
  S = sv; Dx = dx / sv; Dy = dy / sv;
}
// y_retract! (retractions.jl:451-500): (xn, yn) trial, (xb, yb) base point
__device__ __forceinline__ void ineq_yretract(double q, double r, double s, double t, double xb, double yb, double &xn, double &yn) {
  if (q == 0.0 && s == 0.0) { xn = yn; return; }
  if (q == 0.0) {
    const double g1 = -s, g2 = -2.0 * (yb - r), ng = sqrt(g1 * g1 + g2 * g2);
    const double ux = xb - xn + g1 / ng, uy = yb - yn + g2 / ng;
    const double y0 = yn - r;
    const double a = s * uy * uy, b = ux + 2.0 * s * y0 * uy, c = xn + s * y0 * y0 - r;
    const double a1 = -b / (2.0 * a), a2 = sqrt(b * b - 4.0 * a * c) / (2.0 * a);
    const double gam = fmin(a1 + a2, a1 - a2);
    xn += gam * ux; yn += gam * uy;
    return;
  }
  const double rho = sqrt(t);
  const double ex = xn - r, ey = yn - r, dist = sqrt(ex * ex + ey * ey);
  yn = r + rho * ey / dist;
  xn = r + rho * ex / dist;
}

// pb = Dy (Dy v_x - Dx v_y): the x-half operand of PJct' v
__global__ void __launch_bounds__(256) ineq_proj_pre_kernel(IneqDev I, const double *__restrict__ v, double *__restrict__ pb,
                                                            const LargeCtrl *ctrl, int pred) {
  if (pred == 1 && ctrl->status != 0) return;
  const int64_t nx = I.nx;
  for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < nx; j += (int64_t)gridDim.x * 256) {
    const double dy = I.Dy[j];
    pb[j] = dy * (dy * v[j] - I.Dx[j] * v[nx + j]);
  }
}

// the elementwise tail of the projection: (ox, oy) = v - Q Q' v given w_j = sum_rs cpart[rs][j]
__device__ __forceinline__ void ineq_proj_tail(const IneqDev &I, int64_t j, double vx, double vy, const double *cpart, int nsplit,
                                               double &ox, double &oy, double &aa, double &wj) {
  const double s = split_sum(cpart, nsplit, I.nx, j);
  const double dx = I.Dx[j], dy = I.Dy[j];
  aa = dx * vx + dy * vy; wj = s;
  ox = vx - (dx * aa + dy * dy * s);
  oy = vy - (dy * aa - dx * dy * s);
}

// start-up projection of projcg! (projcg.jl:58-62) on the 2n-vector: r = g = P r ; d = -g ; r.r partials -> slot 3
__global__ void __launch_bounds__(256) ineq_cg_init_kernel(IneqDev I, double *__restrict__ r, double *__restrict__ d,
                                                           const double *__restrict__ cpart, int nsplit, double *lp) {
  __shared__ double sh[33];
  const int64_t nx = I.nx;
  double a = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < nx; j += (int64_t)gridDim.x * 256) {
    double ox, oy, aa, wj;
    ineq_proj_tail(I, j, r[j], r[nx + j], cpart, nsplit, ox, oy, aa, wj);
    r[j] = ox; r[nx + j] = oy; d[j] = -1.0 * ox; d[nx + j] = -1.0 * oy;
    a += ox * ox + oy * oy;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[3 * MAXP + blockIdx.x] = a;
}
// gp = P rp ; partials rp.gp (slot 1), gp.gp (slot 2+par)   (projcg.jl:95-99)
__global__ void __launch_bounds__(256) ineq_cg_update2_kernel(IneqDev I, const double *__restrict__ rp, double *__restrict__ gp,
                                                              const double *__restrict__ cpart, int nsplit, double *lp, int par,
                                                              const LargeCtrl *ctrl, int pred) {
  if (pred && ctrl->status != 0) return;
  __shared__ double sh[33];
  const int64_t nx = I.nx;
  double a = 0.0, b = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < nx; j += (int64_t)gridDim.x * 256) {
    const double vx = rp[j], vy = rp[nx + j];
    double ox, oy, aa, wj;
    ineq_proj_tail(I, j, vx, vy, cpart, nsplit, ox, oy, aa, wj);
    gp[j] = ox; gp[nx + j] = oy;
    a += vx * ox + vy * oy; b += ox * ox + oy * oy;
  }
  a = block_sum(a, sh); b = block_sum(b, sh);
  if (threadIdx.x == 0) { lp[1 * MAXP + blockIdx.x] = a; lp[(2 + par) * MAXP + blockIdx.x] = b; }
}
// augmented_hess_lag_vec! (inequality_helper.jl:144-158) on top of a family Hessian action that filled dest_x:
// dest_x += 2 lambda_y q src_x ; dest_y = 2 lambda_y s src_y ; partial src.dest over both halves -> slot 0
__global__ void __launch_bounds__(256) ineq_hess_aug_kernel(IneqDev I, double *__restrict__ dest, const double *__restrict__ src,
                                                            double *lp, const LargeCtrl *ctrl, int pred) {
  if (pred == 1 && ctrl->status != 0) return;
  __shared__ double sh[33];
  const int64_t nx = I.nx;
  double a = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < nx; j += (int64_t)gridDim.x * 256) {
    const double ly2 = 2.0 * I.lamy[j], sx = src[j], sy = src[nx + j];
    const double hx = dest[j] + ly2 * I.q[j] * sx, hy = ly2 * I.s[j] * sy;
    dest[j] = hx; dest[nx + j] = hy;
    a += sx * hx + sy * hy;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[0 * MAXP + blockIdx.x] = a;
}
// ProjPenalty right-hand side with bounds (retractions.jl:369-371): g = bigA [h ; c] + mu g ; dx = 0 ; r = g ; p = 0 ;
// r.r partials -> slot 5
__global__ void __launch_bounds__(256) ineq_pp_rhs_kernel(IneqDev I, double *__restrict__ g, double *__restrict__ dx,
                                                          double *__restrict__ r, double *__restrict__ p,
                                                          const double *__restrict__ cpart, int nsplit, double mu,
                                                          const double *__restrict__ cvh, double *lp) {
  __shared__ double sh[33];
  const int64_t nx = I.nx;
  double a = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < nx; j += (int64_t)gridDim.x * 256) {
    const double s = split_sum(cpart, nsplit, nx, j);
    const double sw = I.S[j] * cvh[j];
    const double gx = (s + I.Dx[j] * sw) + mu * g[j];
    const double gy = mu * g[nx + j] + I.Dy[j] * sw;
    g[j] = gx; g[nx + j] = gy; r[j] = gx; r[nx + j] = gy;
    dx[j] = 0.0; dx[nx + j] = 0.0; p[j] = 0.0; p[nx + j] = 0.0;
    a += gx * gx + gy * gy;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[5 * MAXP + blockIdx.x] = a;
}
// pcg! operator with bounds: z = bigA (bigA' p) + mu p given cpart = J'(J p_x) ; partial p.z (slot 4)
__global__ void __launch_bounds__(256) ineq_pcg_z_kernel(IneqDev I, double *__restrict__ z, const double *__restrict__ p,
                                                         const double *__restrict__ cpart, int nsplit, double *lp,
                                                         const LargeCtrl *ctrl) {
  if (ctrl->pcg_status != 0) return;
  __shared__ double sh[33];
  const int64_t nx = I.nx;
  const double mu = ctrl->mu;
  double a = 0.0;
  for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < nx; j += (int64_t)gridDim.x * 256) {
    const double s = split_sum(cpart, nsplit, nx, j);
    const double px = p[j], py = p[nx + j], Sj = I.S[j], dxj = I.Dx[j], dyj = I.Dy[j];
    const double th = Sj * (dxj * px + dyj * py), sw = Sj * th;
    const double zx = (s + dxj * sw) + mu * px, zy = mu * py + dyj * sw;
    z[j] = zx; z[nx + j] = zy;
    a += px * zx + py * zy;
  }
  a = block_sum(a, sh);
  if (threadIdx.x == 0) lp[4 * MAXP + blockIdx.x] = a;
}
// Jw[a][j] = J[a][j] Dy[j]: the row-scaled operand of the weighted Gram G_w = Jw Jw'  (optimize.jl:288-289 equivalent)
__global__ void __launch_bounds__(256) ineq_scale_cols_kernel(const double *__restrict__ J, int64_t ld, int m, int64_t ncols,
                                                              const double *__restrict__ Dy, double *__restrict__ Jw) {
  const int64_t n2 = ncols >> 1;
  for (int row = blockIdx.y; row < m; row += gridDim.y) {
    const double *src = J + (int64_t)row * ld; double *dst = Jw + (int64_t)row * ld;
    for (int64_t j = (int64_t)blockIdx.x * 256 + threadIdx.x; j < n2; j += (int64_t)gridDim.x * 256) {
      const double2 a = ld_stream2(src + 2 * j), w = *reinterpret_cast<const double2 *>(Dy + 2 * j);
      *reinterpret_cast<double2 *>(dst + 2 * j) = make_double2(a.x * w.x, a.y * w.y);
    }
    if ((ncols & 1) && blockIdx.x == 0 && threadIdx.x == 0) dst[ncols - 1] = src[ncols - 1] * Dy[ncols - 1];
  }
}
// dot-product partials of two vectors -> slot `slot` of lp (host-callback Hessian action: src.dest)
__global__ void __launch_bounds__(256) dot_partials_kernel(int64_t n, const double *__restrict__ a, const double *__restrict__ b,
                                                           double *lp, int slot, const LargeCtrl *ctrl, int pred) {
  if (pred == 1 && ctrl->status != 0) return;
  __shared__ double sh[33];
  double s = 0.0;
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (int64_t)gridDim.x * 256) s += a[i] * b[i];
  s = block_sum(s, sh);
  if (threadIdx.x == 0) lp[(size_t)slot * MAXP + blockIdx.x] = s;
}

}  // namespace lfpsqp
