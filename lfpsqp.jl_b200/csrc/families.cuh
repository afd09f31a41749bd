// families.cuh -- registered device problem families (group-cooperative callbacks).
//
// These replace the closures src/autodiff_generators.jl generates on the CPU (grad! :7-9, jac! :40-42,
// hess_lag_vec! :80-104) with analytic device code.  Every function is called by ALL lanes of the group that
// owns the instance.  Conventions:
//   * inputs were made visible (group sync) by the caller; outputs become visible after the caller's next sync
//   * J is ROW-major with leading dimension ld (row i = gradient of constraint i) == the reference's Jct
//   * jac/jacd only write structural non-zeros when kSparseJac is true (the caller zero-fills first)
//   * f returns the value to every lane
#pragma once
#include "common.cuh"

namespace lfpsqp {

// ---------------------------------------------------------------- Rosenbrock (README.md:18-22)
struct FamRosenbrock {
  static constexpr int kId = LFPSQP_FAM_ROSENBROCK;
  static constexpr bool kSparseJac = true;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n == 2 && m == 0 && p == 0; }
  template <class G> static LFPSQP_DEV double f(const G &, const FamCtx &, const double *x) {
    double a = 1.0 - x[0], b = x[1] - x[0] * x[0];
    return a * a + 100.0 * b * b;
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &, double *out, const double *x) {
    if (g.lane == 0) {
      double b = x[1] - x[0] * x[0];
      out[0] = -2.0 * (1.0 - x[0]) - 400.0 * x[0] * b;
      out[1] = 200.0 * b;
    }
  }
  template <class G> static LFPSQP_DEV void c(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jac(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G> static LFPSQP_DEV void d(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jacd(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &, double *dest, const double *src, const double *x,
                              const double *, const double *) {
    if (g.lane == 0) {
      double h11 = 2.0 - 400.0 * (x[1] - x[0] * x[0]) + 800.0 * x[0] * x[0], h12 = -400.0 * x[0];
      double v0 = src[0], v1 = src[1];
      dest[0] = h11 * v0 + h12 * v1;
      dest[1] = h12 * v0 + 200.0 * v1;
    }
  }
};

// ---------------------------------------------------------------- README equality example (README.md:41-54)
struct FamReadmeEq {
  static constexpr int kId = LFPSQP_FAM_README_EQ;
  static constexpr bool kSparseJac = true;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n >= 1 && m == 1 && p == 0; }
  template <class G> static LFPSQP_DEV double f(const G &g, const FamCtx &fc, const double *x) {
    double s = 0;
    for (int i = g.lane; i < fc.n; i += G::SIZE) s += x[i] * x[i];
    return g.sum(s);
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &fc, double *out, const double *x) {
    for (int i = g.lane; i < fc.n; i += G::SIZE) out[i] = 2.0 * x[i];
  }
  template <class G> static LFPSQP_DEV void c(const G &g, const FamCtx &, double *cv, const double *x) {
    if (g.lane == 0) cv[0] = x[0] - 0.75;
  }
  template <class G>
  static LFPSQP_DEV void jac(const G &g, const FamCtx &, double *J, int, double *cv, const double *x) {
    if (g.lane == 0) { J[0] = 1.0; cv[0] = x[0] - 0.75; }
  }
  template <class G> static LFPSQP_DEV void d(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jacd(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &fc, double *dest, const double *src, const double *,
                              const double *, const double *) {
    for (int i = g.lane; i < fc.n; i += G::SIZE) dest[i] = 2.0 * src[i];
  }
};

// ---------------------------------------------------------------- README inequality example (README.md:57-76)
struct FamReadmeIneq {
  static constexpr int kId = LFPSQP_FAM_README_INEQ;
  static constexpr bool kSparseJac = false;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n >= 1 && m == 0 && p == 1; }
  template <class G> static LFPSQP_DEV double f(const G &g, const FamCtx &fc, const double *x) {
    double s = 0;
    for (int i = g.lane; i < fc.n; i += G::SIZE) s += __ldg(fc.prm + i) * x[i];
    return g.sum(s);
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &fc, double *out, const double *) {
    for (int i = g.lane; i < fc.n; i += G::SIZE) out[i] = __ldg(fc.prm + i);
  }
  template <class G> static LFPSQP_DEV void c(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jac(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G> static LFPSQP_DEV void d(const G &g, const FamCtx &fc, double *dv, const double *x) {
    double s = 0;
    for (int i = g.lane; i < fc.n; i += G::SIZE) s += x[i] * x[i];
    s = g.sum(s);
    if (g.lane == 0) dv[0] = s - 1.0;
  }
  template <class G>
  static LFPSQP_DEV void jacd(const G &g, const FamCtx &fc, double *J, int, double *dv, const double *x) {
    double s = 0;
    for (int i = g.lane; i < fc.n; i += G::SIZE) { double xi = x[i]; J[i] = 2.0 * xi; s += xi * xi; }
    s = g.sum(s);
    if (g.lane == 0) dv[0] = s - 1.0;
  }
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &fc, double *dest, const double *src, const double *,
                              const double *, const double *lam_d) {
    double l2 = 2.0 * lam_d[0];
    for (int i = g.lane; i < fc.n; i += G::SIZE) dest[i] = l2 * src[i];
  }
};

// ---------------------------------------------------------------- Thomson problem (SURVEY 8d C4)
struct FamThomson {
  static constexpr int kId = LFPSQP_FAM_THOMSON;
  static constexpr bool kSparseJac = true;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n >= 6 && n % 3 == 0 && m == n / 3 && p == 0; }
  template <class G> static LFPSQP_DEV double f(const G &g, const FamCtx &fc, const double *x) {
    int N = fc.m; double s = 0;
    for (int i = g.lane; i < N; i += G::SIZE) {
      double xi = x[3 * i], yi = x[3 * i + 1], zi = x[3 * i + 2];
      for (int j = i + 1; j < N; j++) {
        double a = xi - x[3 * j], b = yi - x[3 * j + 1], cc = zi - x[3 * j + 2];
        s += 1.0 / sqrt(a * a + b * b + cc * cc);
      }
    }
    return g.sum(s);
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &fc, double *out, const double *x) {
    int N = fc.m;
    for (int i = g.lane; i < N; i += G::SIZE) {
      double xi = x[3 * i], yi = x[3 * i + 1], zi = x[3 * i + 2], gx = 0, gy = 0, gz = 0;
      for (int j = 0; j < N; j++) {
        if (j == i) continue;
        double a = xi - x[3 * j], b = yi - x[3 * j + 1], cc = zi - x[3 * j + 2];
        double r2 = a * a + b * b + cc * cc, ir3 = 1.0 / (r2 * sqrt(r2));
        gx -= a * ir3; gy -= b * ir3; gz -= cc * ir3;
      }
      out[3 * i] = gx; out[3 * i + 1] = gy; out[3 * i + 2] = gz;
    }
  }
  template <class G> static LFPSQP_DEV void c(const G &g, const FamCtx &fc, double *cv, const double *x) {
    for (int i = g.lane; i < fc.m; i += G::SIZE)
      cv[i] = x[3 * i] * x[3 * i] + x[3 * i + 1] * x[3 * i + 1] + x[3 * i + 2] * x[3 * i + 2] - 1.0;
  }
  template <class G>
  static LFPSQP_DEV void jac(const G &g, const FamCtx &fc, double *J, int ld, double *cv, const double *x) {
    for (int i = g.lane; i < fc.m; i += G::SIZE) {
      double a = x[3 * i], b = x[3 * i + 1], cc = x[3 * i + 2];
      J[(size_t)i * ld + 3 * i] = 2.0 * a; J[(size_t)i * ld + 3 * i + 1] = 2.0 * b; J[(size_t)i * ld + 3 * i + 2] = 2.0 * cc;
      cv[i] = a * a + b * b + cc * cc - 1.0;
    }
  }
  template <class G> static LFPSQP_DEV void d(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jacd(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &fc, double *dest, const double *v, const double *x,
                              const double *lam, const double *) {
    int N = fc.m;
    for (int i = g.lane; i < N; i += G::SIZE) {
      double xi = x[3 * i], yi = x[3 * i + 1], zi = x[3 * i + 2], vx = v[3 * i], vy = v[3 * i + 1], vz = v[3 * i + 2];
      double hx = 0, hy = 0, hz = 0;
      for (int j = 0; j < N; j++) {
        if (j == i) continue;
        double a = xi - x[3 * j], b = yi - x[3 * j + 1], cc = zi - x[3 * j + 2];
        double wa = vx - v[3 * j], wb = vy - v[3 * j + 1], wc = vz - v[3 * j + 2];
        double r2 = a * a + b * b + cc * cc, ir3 = 1.0 / (r2 * sqrt(r2)), ir5 = ir3 / r2;
        double rw = 3.0 * (a * wa + b * wb + cc * wc) * ir5;
        hx += rw * a - wa * ir3; hy += rw * b - wb * ir3; hz += rw * cc - wc * ir3;
      }
      double l2 = 2.0 * lam[i];
      dest[3 * i] = hx + l2 * vx; dest[3 * i + 1] = hy + l2 * vy; dest[3 * i + 2] = hz + l2 * vz;
    }
  }
};

// ---------------------------------------------------------------- diagonal-quadratic constraints (SURVEY 8d C5)
struct FamDiagQuad {
  static constexpr int kId = LFPSQP_FAM_DIAGQUAD;
  static constexpr bool kSparseJac = false;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n >= 1 && m >= 0 && m <= n && p == 0; }
  template <class G> static LFPSQP_DEV double f(const G &g, const FamCtx &fc, const double *x) {
    const double *xt = fc.prm + 2 * (size_t)fc.m * fc.n + fc.m, *w = xt + fc.n;
    double s = 0;
    for (int j = g.lane; j < fc.n; j += G::SIZE) { double t = x[j] - __ldg(xt + j); s += __ldg(w + j) * t * t; }
    return 0.5 * g.sum(s);
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &fc, double *out, const double *x) {
    const double *xt = fc.prm + 2 * (size_t)fc.m * fc.n + fc.m, *w = xt + fc.n;
    for (int j = g.lane; j < fc.n; j += G::SIZE) out[j] = __ldg(w + j) * (x[j] - __ldg(xt + j));
  }
  template <class G> static LFPSQP_DEV void c(const G &g, const FamCtx &fc, double *cv, const double *x) {
    const double *Q = fc.prm, *A = Q + (size_t)fc.m * fc.n, *b = A + (size_t)fc.m * fc.n;
    for (int i = 0; i < fc.m; i++) {
      double s = 0;
      for (int j = g.lane; j < fc.n; j += G::SIZE) {
        double xj = x[j];
        s += (0.5 * __ldg(Q + (size_t)i * fc.n + j) * xj + __ldg(A + (size_t)i * fc.n + j)) * xj;
      }
      s = g.sum(s);
      if (g.lane == 0) cv[i] = s - __ldg(b + i);
    }
  }
  template <class G>
  static LFPSQP_DEV void jac(const G &g, const FamCtx &fc, double *J, int ld, double *cv, const double *x) {
    const double *Q = fc.prm, *A = Q + (size_t)fc.m * fc.n, *b = A + (size_t)fc.m * fc.n;
    for (int i = 0; i < fc.m; i++) {
      double s = 0;
      for (int j = g.lane; j < fc.n; j += G::SIZE) {
        double xj = x[j], q = __ldg(Q + (size_t)i * fc.n + j), a = __ldg(A + (size_t)i * fc.n + j);
        J[(size_t)i * ld + j] = q * xj + a;
        s += (0.5 * q * xj + a) * xj;
      }
      s = g.sum(s);
      if (g.lane == 0) cv[i] = s - __ldg(b + i);
    }
  }
  template <class G> static LFPSQP_DEV void d(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jacd(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &fc, double *dest, const double *v, const double *,
                              const double *lam, const double *) {
    const double *Q = fc.prm, *w = fc.prm + 2 * (size_t)fc.m * fc.n + fc.m + fc.n;
    for (int j = g.lane; j < fc.n; j += G::SIZE) {
      double s = __ldg(w + j);
      for (int i = 0; i < fc.m; i++) s += lam[i] * __ldg(Q + (size_t)i * fc.n + j);
      dest[j] = s * v[j];
    }
  }
};

// ---------------------------------------------------------------- sin system (test/test_retractions.jl:34-54)
struct FamSin {
  static constexpr int kId = LFPSQP_FAM_SIN;
  static constexpr bool kSparseJac = true;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n >= 2 && m >= 0 && 2 * m <= n && p == 0; }
  template <class G> static LFPSQP_DEV double f(const G &g, const FamCtx &fc, const double *x) {
    double s = 0;
    for (int j = g.lane; j < fc.n; j += G::SIZE) { double u = x[j] - __ldg(fc.prm + j); s += u * u; }
    return 0.5 * g.sum(s);
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &fc, double *out, const double *x) {
    for (int j = g.lane; j < fc.n; j += G::SIZE) out[j] = x[j] - __ldg(fc.prm + j);
  }
  template <class G> static LFPSQP_DEV void c(const G &g, const FamCtx &fc, double *cv, const double *x) {
    for (int i = g.lane; i < fc.m; i += G::SIZE) cv[i] = x[2 * i + 1] - sin(x[2 * i]);
  }
  template <class G>
  static LFPSQP_DEV void jac(const G &g, const FamCtx &fc, double *J, int ld, double *cv, const double *x) {
    for (int i = g.lane; i < fc.m; i += G::SIZE) {
      double s, co; sincos(x[2 * i], &s, &co);
      cv[i] = x[2 * i + 1] - s;
      J[(size_t)i * ld + 2 * i + 1] = 1.0; J[(size_t)i * ld + 2 * i] = -co;
    }
  }
  template <class G> static LFPSQP_DEV void d(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jacd(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &fc, double *dest, const double *v, const double *x,
                              const double *lam, const double *) {
    for (int j = g.lane; j < fc.n; j += G::SIZE) {
      double h = v[j];
      if (!(j & 1) && (j >> 1) < fc.m) h += lam[j >> 1] * sin(x[j]) * v[j];
      dest[j] = h;
    }
  }
};

// ---------------------------------------------------------------- bounded quadratic (SURVEY App. D bound-embedding check)
struct FamBoxQuad {
  static constexpr int kId = LFPSQP_FAM_BOXQUAD;
  static constexpr bool kSparseJac = false;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n >= 1 && (m == 0 || m == 1) && p == 0; }
  template <class G> static LFPSQP_DEV double f(const G &g, const FamCtx &fc, const double *x) {
    double s = 0;
    for (int j = g.lane; j < fc.n; j += G::SIZE) { double u = x[j] - __ldg(fc.prm + j); s += u * u; }
    return g.sum(s);
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &fc, double *out, const double *x) {
    for (int j = g.lane; j < fc.n; j += G::SIZE) out[j] = 2.0 * (x[j] - __ldg(fc.prm + j));
  }
  template <class G> static LFPSQP_DEV void c(const G &g, const FamCtx &fc, double *cv, const double *x) {
    if (fc.m == 0) return;
    double s = 0;
    for (int j = g.lane; j < fc.n; j += G::SIZE) s += __ldg(fc.prm + fc.n + j) * x[j];
    s = g.sum(s);
    if (g.lane == 0) cv[0] = s - __ldg(fc.prm + 2 * fc.n);
  }
  template <class G>
  static LFPSQP_DEV void jac(const G &g, const FamCtx &fc, double *J, int, double *cv, const double *x) {
    if (fc.m == 0) return;
    double s = 0;
    for (int j = g.lane; j < fc.n; j += G::SIZE) { double a = __ldg(fc.prm + fc.n + j); J[j] = a; s += a * x[j]; }
    s = g.sum(s);
    if (g.lane == 0) cv[0] = s - __ldg(fc.prm + 2 * fc.n);
  }
  template <class G> static LFPSQP_DEV void d(const G &, const FamCtx &, double *, const double *) {}
  template <class G> static LFPSQP_DEV void jacd(const G &, const FamCtx &, double *, int, double *, const double *) {}
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &fc, double *dest, const double *v, const double *,
                              const double *, const double *) {
    for (int j = g.lane; j < fc.n; j += G::SIZE) dest[j] = 2.0 * v[j];
  }
};

// ---------------------------------------------------------------- dense QCQP given by data (lfpsqp_qcqp)
// f = 1/2 x'Px + q.x + r ; c_i = 1/2 x'Qc_i x + Ac_i.x - bc_i ; d_k = 1/2 x'Qd_k x + Ad_k.x - bd_k.
// The matrices are symmetric, so (M v)_j = sum_i M_ij v_i reads row i coalesced across the lanes (lane = column j),
// through L2 with __ldg.  A NULL array is skipped, not read as zeros; the test is group-uniform (the descriptor is a
// kernel parameter).  A quadratic's value is sum_j (0.5 (Mx)_j + a_j) x_j: with M = 2I and a = NULL every term is
// x_j x_j exactly, which is what makes the README families' encodings give their registered results bit for bit.
struct FamQCQP {
  static constexpr int kId = LFPSQP_FAM_QCQP;
  static constexpr bool kSparseJac = false;
  static __host__ bool valid(int64_t n, int64_t m, int64_t p) { return n >= 1 && m >= 0 && p >= 0; }
  // this instance's copy of one array (NULL stays NULL)
  static LFPSQP_DEV const double *arr(const FamCtx &fc, const double *base, int64_t stride) {
    return base ? base + fc.k * stride : nullptr;
  }
  // (M v)_j of a symmetric n x n matrix
  static LFPSQP_DEV double mv(const double *M, const double *v, int n, int j) {
    double s = 0;
#pragma unroll 4
    for (int i = 0; i < n; i++) s += __ldg(M + (size_t)i * n + j) * v[i];
    return s;
  }
  // 1/2 x'Mx + a.x - b (M, a, b may be NULL, not both M and a); with row != NULL also writes the gradient Mx + a
  template <class G>
  static LFPSQP_DEV double quad(const G &g, int n, const double *M, const double *a, const double *b, double *row,
                                const double *x) {
    double s = 0;
    for (int j = g.lane; j < n; j += G::SIZE) {
      double gj, w;
      if (M) {
        const double u = mv(M, x, n, j);
        gj = u; w = 0.5 * u;
        if (a) { const double aj = __ldg(a + j); gj += aj; w += aj; }
      } else {
        gj = w = __ldg(a + j);
      }
      if (row) row[j] = gj;
      s += w * x[j];
    }
    s = g.sum(s);
    return b ? s - __ldg(b) : s;
  }
  template <class G> static LFPSQP_DEV double f(const G &g, const FamCtx &fc, const double *x) {
    const double *P = arr(fc, fc.qp.P, fc.qp.P_stride), *q = arr(fc, fc.qp.q, fc.qp.q_stride);
    const double *r = arr(fc, fc.qp.r, fc.qp.r_stride);
    const double v = (P || q) ? quad(g, fc.n, P, q, nullptr, nullptr, x) : 0.0;
    return r ? v + __ldg(r) : v;
  }
  template <class G> static LFPSQP_DEV void grad(const G &g, const FamCtx &fc, double *out, const double *x) {
    const double *P = arr(fc, fc.qp.P, fc.qp.P_stride), *q = arr(fc, fc.qp.q, fc.qp.q_stride);
    for (int j = g.lane; j < fc.n; j += G::SIZE) {
      double gj = 0.0;
      if (P) { gj = mv(P, x, fc.n, j); if (q) gj += __ldg(q + j); }
      else if (q) gj = __ldg(q + j);
      out[j] = gj;
    }
  }
  // rows of one constraint block (cnt quadratics): values into cv, gradients into J (row stride ld) when J != NULL
  template <class G>
  static LFPSQP_DEV void block(const G &g, const FamCtx &fc, int cnt, const double *Q, int64_t Qs, const double *A,
                               int64_t As, const double *b, int64_t bs, double *J, int ld, double *cv, const double *x) {
    const int n = fc.n;
    Q = arr(fc, Q, Qs); A = arr(fc, A, As); b = arr(fc, b, bs);
    for (int i = 0; i < cnt; i++) {
      const double v = quad(g, n, Q ? Q + (size_t)i * n * n : nullptr, A ? A + (size_t)i * n : nullptr,
                            b ? b + i : nullptr, J ? J + (size_t)i * ld : nullptr, x);
      if (g.lane == 0) cv[i] = v;
    }
  }
  template <class G> static LFPSQP_DEV void c(const G &g, const FamCtx &fc, double *cv, const double *x) {
    block(g, fc, fc.m, fc.qp.Qc, fc.qp.Qc_stride, fc.qp.Ac, fc.qp.Ac_stride, fc.qp.bc, fc.qp.bc_stride, nullptr, 0, cv, x);
  }
  template <class G>
  static LFPSQP_DEV void jac(const G &g, const FamCtx &fc, double *J, int ld, double *cv, const double *x) {
    block(g, fc, fc.m, fc.qp.Qc, fc.qp.Qc_stride, fc.qp.Ac, fc.qp.Ac_stride, fc.qp.bc, fc.qp.bc_stride, J, ld, cv, x);
  }
  template <class G> static LFPSQP_DEV void d(const G &g, const FamCtx &fc, double *dv, const double *x) {
    block(g, fc, fc.p, fc.qp.Qd, fc.qp.Qd_stride, fc.qp.Ad, fc.qp.Ad_stride, fc.qp.bd, fc.qp.bd_stride, nullptr, 0, dv, x);
  }
  template <class G>
  static LFPSQP_DEV void jacd(const G &g, const FamCtx &fc, double *J, int ld, double *dv, const double *x) {
    block(g, fc, fc.p, fc.qp.Qd, fc.qp.Qd_stride, fc.qp.Ad, fc.qp.Ad_stride, fc.qp.bd, fc.qp.bd_stride, J, ld, dv, x);
  }
  // dest = (P + sum_i lam_i Qc_i + sum_k lam_d_k Qd_k) v, one pass over every matrix's rows
  template <class G>
  static LFPSQP_DEV void hess(const G &g, const FamCtx &fc, double *dest, const double *v, const double *,
                              const double *lam, const double *lam_d) {
    const int n = fc.n;
    const size_t nn = (size_t)n * n;
    const double *P = arr(fc, fc.qp.P, fc.qp.P_stride), *Qc = arr(fc, fc.qp.Qc, fc.qp.Qc_stride);
    const double *Qd = arr(fc, fc.qp.Qd, fc.qp.Qd_stride);
    for (int j = g.lane; j < n; j += G::SIZE) {
      double s = P ? mv(P, v, n, j) : 0.0;
      if (Qc) for (int i = 0; i < fc.m; i++) s += lam[i] * mv(Qc + i * nn, v, n, j);
      if (Qd) for (int k = 0; k < fc.p; k++) s += lam_d[k] * mv(Qd + k * nn, v, n, j);
      dest[j] = s;
    }
  }
};

}  // namespace lfpsqp
