// batched_warp.cuh -- one warp per SQP instance, the whole LFPSQP driver on device, state in shared memory.
//
// Replaces, for small dense instances, the reference's L2 driver and L1 kernels (SURVEY.md section 8a):
//   driver loop            src/optimize.jl:257-435          -> Solver::run
//   slack wrapper          src/optimize.jl:13-71            -> *_aux callbacks
//   ksvd!/kgemv! projector src/la_helper.jl:8-44, optimize.jl:288-317 -> factor()/project()  (Gram J W J' + Cholesky)
//   multipliers            optimize.jl:331-343, inequality_helper.jl:286-308 -> by-product of project()
//   projcg!                src/projcg.jl:40-121             -> projcg()
//   armijo!                src/linesearch.jl:32-89          -> armijo()
//   retract! (4 methods)   src/retractions.jl:61-72, :75-177, :265-441, pcg! :179-246, y_retract! :451-500
//   bound embedding        src/inequality_helper.jl:92-271  -> ineq_* / fullJ_* operators
//
// SVD -> Gram/Cholesky mapping (SURVEY.md App. B): U U' = PJct G^-1 PJct',  G = J diag(w) J' with w = 1 (no
// bounds) or Dy^2 (bounds);  V S^-1 U' = G^-1 PJct';  NR runs in the Cholesky-QR basis Q = PJct L^-T, D0 = L^-1.
#pragma once
#include "common.cuh"
#include "families.cuh"

namespace lfpsqp {

// Per-instance shared-memory layout (in doubles).  Host and device compute the same offsets.
struct WarpLayout {
  int n, m, p, NA, ME, N, M, ineq, use_nr, use_exact;
  int o_ex[4], o_V;
  int o_x, o_xnew, o_xtil, o_g, o_d, o_nd, o_w[5], o_J, o_G, o_cval, o_lam, o_tm, o_cvaug, o_u, o_scr, o_Dx, o_Dy, o_S,
      o_lamy, o_D, o_nr, total;
  __host__ __device__ WarpLayout(int n_, int m_, int p_, int ineq_, int use_nr_, int use_exact_ = 0) {
    n = n_; m = m_; p = p_; ineq = ineq_; use_nr = use_nr_; use_exact = use_exact_;
    NA = n + p; ME = m + p; N = ineq ? 2 * NA : NA; M = ineq ? ME + NA : ME;
    int o = 0;
    auto take = [&](int k) { int r = o; o += k; return r; };
    o_x = take(N); o_xnew = take(N); o_xtil = take(N); o_g = take(N); o_d = take(N); o_nd = take(N);
    for (int i = 0; i < 5; i++) o_w[i] = take(N);
    o_J = take(ME * NA); o_G = take(ME * ME); o_cval = take(ME); o_lam = take(ME); o_tm = take(M > 0 ? M : 1);
    o_cvaug = take(M > 0 ? M : 1); o_u = take(ME > 0 ? ME : 1); o_scr = take(NA);
    if (ineq) { o_Dx = take(NA); o_Dy = take(NA); o_S = take(NA); o_lamy = take(NA); }
    else { o_Dx = o_Dy = o_S = o_lamy = 0; }
    if (use_nr && ME > 0) { o_D = take(ME * ME); o_nr = take(3 * ME); } else { o_D = o_nr = 0; }
    for (int i = 0; i < 4; i++) o_ex[i] = use_exact ? take(N) : 0;
    o_V = take(ME * ME + ME);   // eigenvectors + eigenvalues of G (rank-deficient fallback)
    total = (o + 1) & ~1;
  }
};

template <class Fam, class G>
struct Solver {
  const G g;
  const WarpLayout &L;
  const lfpsqp_params &prm;
  FamCtx fc;
  double *sm;  // this instance's workspace
  // bound data (inequality_helper.jl:1-8), shared by the batch; kind: 0 line, 1 parabola, 2 circle
  const double *bkind, *bq, *br, *bs, *bt;
  const int n, m, p, NA, ME, N, M;
  const bool ineq;
  lfpsqp_stats st;
  int status;
  int rank;      // numerical rank of the (projected) Jacobian, optimize.jl:297-302
  bool pinv;     // Gm holds the truncated pseudo-inverse G^+ instead of the Cholesky factor
  double ls_alpha;        // step length returned by the last armijo! / exact_linesearch! (linesearch.jl:88, :338)
  int ls_it1, ls_it2;     // tot_iter1 / tot_iter2 of the last line search

  double *x, *xnew, *xtil, *gr, *d, *nd, *w0, *w1, *w2, *w3, *w4, *J, *Gm, *cval, *lam, *tm, *cvaug, *ub, *scr, *Dx, *Dy,
      *S, *lamy, *Dnr, *nrt;

  LFPSQP_DEV Solver(const G &g_, const WarpLayout &L_, const lfpsqp_params &prm_, double *sm_, const double *bnd)
      : g(g_), L(L_), prm(prm_), sm(sm_), n(L_.n), m(L_.m), p(L_.p), NA(L_.NA), ME(L_.ME), N(L_.N), M(L_.M),
        ineq(L_.ineq != 0) {
    x = sm + L.o_x; xnew = sm + L.o_xnew; xtil = sm + L.o_xtil; gr = sm + L.o_g; d = sm + L.o_d; nd = sm + L.o_nd;
    w0 = sm + L.o_w[0]; w1 = sm + L.o_w[1]; w2 = sm + L.o_w[2]; w3 = sm + L.o_w[3]; w4 = sm + L.o_w[4];
    J = sm + L.o_J; Gm = sm + L.o_G; cval = sm + L.o_cval; lam = sm + L.o_lam; tm = sm + L.o_tm; cvaug = sm + L.o_cvaug;
    ub = sm + L.o_u; scr = sm + L.o_scr; Dx = sm + L.o_Dx; Dy = sm + L.o_Dy; S = sm + L.o_S; lamy = sm + L.o_lamy;
    Dnr = sm + L.o_D; nrt = sm + L.o_nr;
    bkind = bnd; bq = bnd + NA; br = bnd + 2 * NA; bs = bnd + 3 * NA; bt = bnd + 4 * NA;
    fc.n = n; fc.m = m; fc.p = p; fc.prm = nullptr;
    status = 0; rank = ME; pinv = false;
  }

  // ------------------------------------------------------------ small vector helpers (all end with a group sync)
  // the reductions end with a group barrier: a later write to the operands by another lane is then ordered after
  // every lane's reads by the memory model (racecheck-clean), not merely by the shuffle's convergence
  LFPSQP_DEV double dot(const double *a, const double *b, int len) const {
    double s = 0;
    for (int i = g.lane; i < len; i += G::SIZE) s += a[i] * b[i];
    s = g.sum(s);
    g.sync();
    return s;
  }
  LFPSQP_DEV double norminf(const double *a, int len) const {
    double s = 0;
    for (int i = g.lane; i < len; i += G::SIZE) s = pmax(fabs(a[i]), s);
    s = g.maxabs(s);
    g.sync();
    return s;
  }
  LFPSQP_DEV void copy(double *dst, const double *src, int len) const {
    for (int i = g.lane; i < len; i += G::SIZE) dst[i] = src[i];
    g.sync();
  }
  LFPSQP_DEV void fill(double *dst, double v, int len) const {
    for (int i = g.lane; i < len; i += G::SIZE) dst[i] = v;
    g.sync();
  }
  // out[a] = sum_j Jm[a][j] * v[j], a < ME  (one pass over the ME x NA row-major Jacobian)
  LFPSQP_DEV void rowdots(double *out, const double *v) const {
    if (ME >= 16) {  // one row per lane, serial over columns
      for (int a = g.lane; a < ME; a += G::SIZE) {
        const double *row = J + (size_t)a * NA; double s = 0;
        for (int j = 0; j < NA; j++) s += row[j] * v[j];
        out[a] = s;
      }
    } else {
      for (int a = 0; a < ME; a++) {
        const double *row = J + (size_t)a * NA; double s = 0;
        for (int j = g.lane; j < NA; j += G::SIZE) s += row[j] * v[j];
        s = g.sum(s);
        if (g.lane == 0) out[a] = s;
      }
    }
    g.sync();
  }
  // (J' u)_j
  LFPSQP_DEV double coldot(const double *u, int j) const {
    double s = 0;
    for (int a = 0; a < ME; a++) s += J[(size_t)a * NA + j] * u[a];
    return s;
  }

  // ------------------------------------------------------------ problem callbacks on the slack-augmented problem
  LFPSQP_DEV double f_aux(const double *xx) { st.f_evals++; return Fam::f(g, fc, xx); }          // optimize.jl:38-40
  LFPSQP_DEV void grad_aux(double *out, const double *xx) const {
    Fam::grad(g, fc, out, xx);  // entries n..N-1 of the gradient stay 0 (optimize.jl:191)
    g.sync();
  }
  LFPSQP_DEV void c_aux(double *cv, const double *xx) const {                                     // optimize.jl:42-51
    if (m > 0) Fam::c(g, fc, cv, xx);
    if (p > 0) {
      Fam::d(g, fc, cv + m, xx);
      g.sync();
      for (int k = g.lane; k < p; k += G::SIZE) cv[m + k] -= xx[n + k];
    }
    g.sync();
  }
  LFPSQP_DEV void jac_aux(double *cv, const double *xx) const {  // jac!(Jc, cval, x): fills J and cval
    if (Fam::kSparseJac || p > 0) fill(J, 0.0, ME * NA);
    if (m > 0) Fam::jac(g, fc, J, NA, cv, xx);
    if (p > 0) {
      Fam::jacd(g, fc, J + (size_t)m * NA, NA, cv + m, xx);
      g.sync();
      for (int k = g.lane; k < p; k += G::SIZE) { J[(size_t)(m + k) * NA + n + k] = -1.0; cv[m + k] -= xx[n + k]; }
    }
    g.sync();
  }
  // Lagrangian Hessian action at the current (x, lam, lamy): hess_lag_vec! (autodiff_generators.jl:80-104) wrapped by
  // the slack layer and by augmented_hess_lag_vec! (inequality_helper.jl:144-158)
  LFPSQP_DEV void hess_aux(double *dest, const double *src) const {
    Fam::hess(g, fc, dest, src, x, lam, lam + m);
    for (int k = g.lane; k < p; k += G::SIZE) dest[n + k] = 0.0;
    g.sync();
    if (ineq) {
      for (int j = g.lane; j < NA; j += G::SIZE) {
        double ly2 = 2.0 * lamy[j];
        dest[j] += ly2 * bq[j] * src[j];
        dest[NA + j] = ly2 * bs[j] * src[NA + j];
      }
      g.sync();
    }
  }

  // ------------------------------------------------------------ bound embedding (inequality_helper.jl)
  LFPSQP_DEV void generate_initial_y(double *xx) const {  // :92-109
    for (int j = g.lane; j < NA; j += G::SIZE) {
      int kind = (int)bkind[j]; double xv = xx[j], y;
      if (kind == 0) y = xv;
      else if (kind == 1) y = sqrt(fmax(-(xv - bt[j]) / bs[j], 0.0)) + br[j];
      else y = sqrt(fmax(bt[j] - (xv - br[j]) * (xv - br[j]), 0.0)) + br[j];
      xx[NA + j] = y;
    }
    g.sync();
  }
  LFPSQP_DEV void calculate_h(double *out, const double *xx) const {  // :112-122
    for (int j = g.lane; j < NA; j += G::SIZE) {
      double q = bq[j], s = bs[j], r = br[j], dx = xx[j] - r, dy = xx[NA + j] - r;
      out[j] = q * (dx * dx) + (1.0 - q * q) * xx[j] + s * (dy * dy) - (1.0 - s * s) * xx[NA + j] - bt[j];
    }
    g.sync();
  }
  LFPSQP_DEV void inequality_gradient(const double *xx) const {  // :125-141
    for (int j = g.lane; j < NA; j += G::SIZE) {
      double q = bq[j], s = bs[j], r = br[j];
      double dx = 2.0 * q * (xx[j] - r) + (q == 0.0 ? 1.0 : 0.0);
      double dy = 2.0 * s * (xx[NA + j] - r) - (s == 0.0 ? 1.0 : 0.0);
      double sv = sqrt(dx * dx + dy * dy);
      S[j] = sv; Dx[j] = dx / sv; Dy[j] = dy / sv;
    }
    g.sync();
  }
  LFPSQP_DEV void y_retract(double *xn, const double *xb) const {  // retractions.jl:451-500
    for (int j = g.lane; j < NA; j += G::SIZE) {
      int kind = (int)bkind[j];
      if (kind == 0) { xn[j] = xn[NA + j]; }
      else if (kind == 1) {
        double s = bs[j], r = br[j];
        double g1 = -s, g2 = -2.0 * (xb[NA + j] - r), ng = sqrt(g1 * g1 + g2 * g2);
        double ux = xb[j] - xn[j] + g1 / ng, uy = xb[NA + j] - xn[NA + j] + g2 / ng;
        double yn = xn[NA + j] - r;
        double a = s * uy * uy, b = ux + 2.0 * s * yn * uy, c = xn[j] + s * yn * yn - r;
        double a1 = -b / (2.0 * a), a2 = sqrt(b * b - 4.0 * a * c) / (2.0 * a);
        double gam = fmin(a1 + a2, a1 - a2);
        xn[j] += gam * ux; xn[NA + j] += gam * uy;
      } else {
        double c = br[j], rho = sqrt(bt[j]);
        double ex = xn[j] - c, ey = xn[NA + j] - c, dist = sqrt(ex * ex + ey * ey);
        xn[NA + j] = c + rho * ey / dist;
        xn[j] = c + rho * ex / dist;
      }
    }
    g.sync();
  }
  // fulljac * v (retractions.jl:324): J v, or bigA' v (inequality_helper.jl:254-271)
  LFPSQP_DEV void fullJ_mul(double *out, const double *v) const {
    if (ineq) {
      for (int j = g.lane; j < NA; j += G::SIZE) out[j] = S[j] * (Dx[j] * v[j] + Dy[j] * v[NA + j]);
      rowdots(out + NA, v);
    } else rowdots(out, v);
  }
  // dest = a * fulljac' w + b * dest : J' w, or bigA w (inequality_helper.jl:215-251)
  LFPSQP_DEV void fullJ_mulT(double *dest, const double *w, double a, double b) const {
    if (ineq) {
      for (int j = g.lane; j < NA; j += G::SIZE) {
        double t = coldot(w + NA, j), sw = S[j] * w[j];
        dest[j] = a * (t + Dx[j] * sw) + (b == 0.0 ? 0.0 : b * dest[j]);
        dest[NA + j] = (b == 0.0 ? 0.0 : b * dest[NA + j]) + a * Dy[j] * sw;
      }
    } else {
      for (int j = g.lane; j < NA; j += G::SIZE) dest[j] = a * coldot(w, j) + (b == 0.0 ? 0.0 : b * dest[j]);
    }
    g.sync();
  }

  // ------------------------------------------------------------ Gram + Cholesky (replaces ksvd!, optimize.jl:288-302)
  // G = J diag(w) J', w = Dy^2 with bounds (PJct'PJct, App. B) else 1; in-place lower Cholesky. false = rank deficient.
  LFPSQP_DEV double gram() {   // Gm (lower) = J diag(w) J' ; returns max diag
    double maxdiag = 0.0;
    for (int a = 0; a < ME; a++) {
      for (int b = 0; b <= a; b++) {
        const double *ra = J + (size_t)a * NA, *rb = J + (size_t)b * NA; double s = 0;
        if (ineq) for (int j = g.lane; j < NA; j += G::SIZE) { double wy = Dy[j]; s += ra[j] * (wy * wy) * rb[j]; }
        else for (int j = g.lane; j < NA; j += G::SIZE) s += ra[j] * rb[j];
        s = g.sum(s);
        if (g.lane == 0) Gm[a * ME + b] = s;
        if (a == b) maxdiag = fmax(maxdiag, s);
      }
    }
    g.sync();
    return maxdiag;
  }
  LFPSQP_DEV bool factor() {
    st.factorizations++;
    rank = ME; pinv = false;
    const double maxdiag = gram();
    const double thresh = fmax(prm.eps_rank * prm.eps_rank, 1e-14 * maxdiag);
    for (int k = 0; k < ME; k++) {
      for (int i = k + g.lane; i < ME; i += G::SIZE) {
        double s = Gm[i * ME + k];
        for (int t = 0; t < k; t++) s -= Gm[i * ME + t] * Gm[k * ME + t];
        Gm[i * ME + k] = s;
      }
      g.sync();
      double piv = Gm[k * ME + k];
      if (!(piv > thresh)) { factor_rank_deficient(); return true; }
      double rinv = 1.0 / sqrt(piv);
      g.sync();
      for (int i = k + g.lane; i < ME; i += G::SIZE) Gm[i * ME + k] = (i == k) ? sqrt(piv) : Gm[i * ME + k] * rinv;
      g.sync();
    }
    return true;
  }
  // Rank-deficient Jacobian (optimize.jl:297-302: rank = #{sigma_j >= eps_rank}, projector on U[:,1:rank], multipliers
  // zeroed beyond rank, :335-340).  Gram-form equivalent: G = V diag(sigma^2) V' by cyclic Jacobi rotations, and the
  // truncated pseudo-inverse G^+ = V_r diag(1/sigma_r^2) V_r' takes the place of (L L')^-1 in every solve:
  //   U_r U_r' = PJct G^+ PJct' ,  lambda = V Sigma_r^-1 U_r'(-g) = G^+ PJct'(-g).
  // Eigenvalues below max(eps_rank^2, 1e-13 * sigma_max^2) count as zero (the Gram form cannot see singular values
  // below ~3e-7 * sigma_max; the SVD-based reference resolves them down to eps_rank).
  LFPSQP_DEV void factor_rank_deficient() {
    double *V = sm + L.o_V, *ev = V + ME * ME;
    gram();
    for (int e = g.lane; e < ME * ME; e += G::SIZE) {       // symmetrise, V = I
      int a = e / ME, b = e % ME;
      if (b > a) Gm[a * ME + b] = Gm[b * ME + a];
      V[e] = (a == b) ? 1.0 : 0.0;
    }
    g.sync();
    for (int sweep = 0; sweep < 30; sweep++) {
      double off = 0.0, dg = 0.0;
      for (int e = g.lane; e < ME * ME; e += G::SIZE) { double v = Gm[e]; if (e / ME != e % ME) off += v * v; else dg += v * v; }
      off = g.sum(off); dg = g.sum(dg);
      if (off <= 1e-30 * dg || off == 0.0) break;
      for (int pq = 0; pq < ME - 1; pq++)
        for (int q = pq + 1; q < ME; q++) {
          const double apq = Gm[pq * ME + q];
          if (apq == 0.0) continue;                          // uniform: every lane reads the same value
          const double app = Gm[pq * ME + pq], aqq = Gm[q * ME + q];
          const double theta = (aqq - app) / (2.0 * apq);
          const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
          const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
          g.sync();
          for (int k = g.lane; k < ME; k += G::SIZE) {       // columns p, q of A and V
            double akp = Gm[k * ME + pq], akq = Gm[k * ME + q];
            Gm[k * ME + pq] = c * akp - sn * akq; Gm[k * ME + q] = sn * akp + c * akq;
            double vkp = V[k * ME + pq], vkq = V[k * ME + q];
            V[k * ME + pq] = c * vkp - sn * vkq; V[k * ME + q] = sn * vkp + c * vkq;
          }
          g.sync();
          for (int k = g.lane; k < ME; k += G::SIZE) {       // rows p, q of A
            double apk = Gm[pq * ME + k], aqk = Gm[q * ME + k];
            Gm[pq * ME + k] = c * apk - sn * aqk; Gm[q * ME + k] = sn * apk + c * aqk;
          }
          g.sync();
        }
    }
    double lmax = 0.0;
    for (int k = 0; k < ME; k++) lmax = fmax(lmax, Gm[k * ME + k]);
    const double thr = fmax(prm.eps_rank * prm.eps_rank, 1e-13 * lmax);
    int r = 0;
    for (int k = 0; k < ME; k++) { double lv = Gm[k * ME + k]; if (lv >= thr) r++; }
    g.sync();
    for (int k = g.lane; k < ME; k += G::SIZE) { double lv = Gm[k * ME + k]; ev[k] = (lv >= thr) ? 1.0 / lv : 0.0; }
    g.sync();
    for (int e = g.lane; e < ME * ME; e += G::SIZE) {       // G^+ = V diag(ev) V'
      int a = e / ME, b = e % ME; double s2 = 0.0;
      for (int k = 0; k < ME; k++) s2 += V[a * ME + k] * ev[k] * V[b * ME + k];
      Gm[e] = s2;
    }
    g.sync();
    rank = r; pinv = true;
  }
  // u <- G^-1 u : Cholesky solves, or the truncated pseudo-inverse when the Jacobian is rank deficient
  LFPSQP_DEV void solveG(double *u) const {
    if (!pinv) { solveL(u); solveLt(u); return; }
    double *tmp = sm + L.o_V + ME * ME;   // the eigenvalue slots are free once G^+ is formed
    for (int a = g.lane; a < ME; a += G::SIZE) { double s2 = 0.0; for (int b = 0; b < ME; b++) s2 += Gm[a * ME + b] * u[b]; tmp[a] = s2; }
    g.sync();
    for (int a = g.lane; a < ME; a += G::SIZE) u[a] = tmp[a];
    g.sync();
  }
  LFPSQP_DEV void solveL(double *u) const {  // u <- L^-1 u
    for (int k = 0; k < ME; k++) {
      g.sync();
      double uk = u[k] / Gm[k * ME + k];
      g.sync();
      if (g.lane == 0) u[k] = uk;
      for (int i = k + 1 + g.lane; i < ME; i += G::SIZE) u[i] -= Gm[i * ME + k] * uk;
    }
    g.sync();
  }
  LFPSQP_DEV void solveLt(double *u) const {  // u <- L^-T u
    for (int k = ME - 1; k >= 0; k--) {
      g.sync();
      double uk = u[k] / Gm[k * ME + k];
      g.sync();
      if (g.lane == 0) u[k] = uk;
      for (int i = g.lane; i < k; i += G::SIZE) u[i] -= Gm[k * ME + i] * uk;
    }
    g.sync();
  }

  // v <- v - Q Q' v : tangent projection (optimize.jl:306-307 / :316-317, projcg.jl:59-60,:96-97).
  // With want_mult the multipliers fall out (optimize.jl:331-343, calculate_lambda_kkt! inequality_helper.jl:286-308).
  LFPSQP_DEV void project(double *v, bool want_mult) {
    if (ineq) {
      for (int j = g.lane; j < NA; j += G::SIZE) {
        double vx = v[j], vy = v[NA + j], dx = Dx[j], dy = Dy[j];
        tm[j] = dx * vx + dy * vy;            // (Q'v)[1:n]
        scr[j] = dy * (dy * vx - dx * vy);    // PJct' v = J * scr
      }
      g.sync();
      if (ME > 0) { rowdots(ub, scr); solveG(ub); }
      for (int j = g.lane; j < NA; j += G::SIZE) {
        double wj = (ME > 0) ? coldot(ub, j) : 0.0, dx = Dx[j], dy = Dy[j], a = tm[j];
        v[j] -= dx * a + dy * dy * wj;
        v[NA + j] -= dy * a - dx * dy * wj;
        if (want_mult) lamy[j] = (-1.0 * dx / S[j]) * wj + a / S[j];
      }
      if (want_mult) for (int a = g.lane; a < ME; a += G::SIZE) lam[a] = ub[a];
      g.sync();
    } else if (ME > 0) {
      rowdots(ub, v); solveG(ub);
      for (int j = g.lane; j < NA; j += G::SIZE) v[j] -= coldot(ub, j);
      if (want_mult) for (int a = g.lane; a < ME; a += G::SIZE) lam[a] = ub[a];
      g.sync();
    }
  }

  // ------------------------------------------------------------ projcg! (projcg.jl:40-121), c = 0 as the driver passes
  // solution in nd; returns iterations, nr_out = final projected residual norm (Inf on negative curvature)
  LFPSQP_DEV int projcg(const double *b, int clen, double tol, int64_t maxit, double *nr_out) {
    double *xs = nd, *r = w0, *dc = w1, *Ad = w2, *rp = w3, *gp = w4;
    for (int i = g.lane; i < N; i += G::SIZE) { xs[i] = 0.0; r[i] = -b[i]; }   // :55-57 with x = U*0
    g.sync();
    project(r, false);                                                          // :58-61 (g = r)
    for (int i = g.lane; i < N; i += G::SIZE) dc[i] = -1.0 * r[i];
    g.sync();
    int i = 0; double nr = INFINITY;
    int64_t lim = (int64_t)N + clen; if (maxit < lim) lim = maxit;
    while (i < lim) {
      i++;
      hess_aux(Ad, dc);                                                         // :74
      double dAd = dot(dc, Ad, N);
      if (dAd <= 0.0) {                                                         // :77-82
        double nrm = sqrt(dot(dc, dc, N));
        for (int k = g.lane; k < N; k += G::SIZE) xs[k] = dc[k] / nrm;
        g.sync();
        st.projcg_iters += i; st.projcg_negcurv++;
        *nr_out = INFINITY; return i;
      }
      double rg = dot(r, r, N);                                                 // r == g after every projection
      if (rg <= 0.0) break;                                                     // :87-89
      double alpha = rg / dAd;
      for (int k = g.lane; k < N; k += G::SIZE) {
        xs[k] += alpha * dc[k];
        double t = r[k] + alpha * Ad[k];
        rp[k] = t; gp[k] = t;
      }
      g.sync();
      project(gp, false);                                                       // :95-97
      double beta = dot(rp, gp, N) / rg;
      double s = 0;
      for (int k = g.lane; k < N; k += G::SIZE) {
        double gk = gp[k];
        dc[k] = beta * dc[k] - gk; r[k] = gk; s += gk * gk;
      }
      nr = sqrt(g.sum(s));
      g.sync();
      if (nr < tol) break;                                                      // :107-111
    }
    st.projcg_iters += i;
    *nr_out = nr; return i;
  }

  // ------------------------------------------------------------ pcg! (retractions.jl:179-246), no preconditioner
  LFPSQP_DEV int pcg(double mu, double *xs, double *r, double *pv, double *z, double tol, int64_t maxiter, int *iters) {
    double norm_res = INFINITY, rho = 1.0;
    fill(pv, 0.0, N);
    int i = 0;
    while (norm_res > tol && i < maxiter) {
      double rho_prev = rho; rho = dot(r, r, N);          // z = r (M! = copy)
      double beta = rho / rho_prev;
      for (int k = g.lane; k < N; k += G::SIZE) pv[k] = r[k] + beta * pv[k];
      g.sync();
      fullJ_mul(tm, pv);
      for (int k = g.lane; k < N; k += G::SIZE) z[k] = pv[k];
      g.sync();
      fullJ_mulT(z, tm, 1.0, mu);                         // z = J'(J p) + mu p
      double alpha = rho / dot(pv, z, N);
      double s = 0;
      for (int k = g.lane; k < N; k += G::SIZE) {
        xs[k] += alpha * pv[k];
        double rk = r[k] - alpha * z[k];
        r[k] = rk; s += rk * rk;
      }
      norm_res = sqrt(g.sum(s));
      g.sync();
      i++;
    }
    *iters = i;
    return (i == maxiter) ? 1 : 0;
  }

  // ------------------------------------------------------------ retract!(::ProjPenalty) (retractions.jl:265-441)
  LFPSQP_DEV int retract_pp(int *it1, int *it2) {
    double *r = w0, *pv = w1, *z = w2, *dx = w3, *gv = w4;
    int flag = 0;
    copy(xnew, xtil, N);
    double mu = prm.mu0;
    int i = 0, pcg_total = 0;
    while (i < prm.maxiter_retract) {
      jac_aux(cval, xnew);                                              // :340
      double curtol = norminf(cval, ME);
      if (ineq) {
        inequality_gradient(xnew);                                      // :344 (shared idecomp: driver recomputes)
        calculate_h(cvaug, xnew);                                       // :350
        curtol = pmax(curtol, norminf(cvaug, M));                       // :352 incl. the stale tail of cvalaug
      }
      for (int a = g.lane; a < ME; a += G::SIZE) cvaug[M - ME + a] = cval[a];   // :356
      g.sync();
      if (curtol < prm.eps_c) break;                                    // :359-361
      for (int k = g.lane; k < N; k += G::SIZE) gv[k] = xnew[k] - xtil[k];
      g.sync();
      double prev_obj = dot(cvaug, cvaug, M) + mu * dot(gv, gv, N);     // :366
      fullJ_mulT(gv, cvaug, 1.0, mu);                                   // :369
      for (int k = g.lane; k < N; k += G::SIZE) { dx[k] = 0.0; r[k] = gv[k]; }
      g.sync();
      int pcg_i = 0;
      int pcg_flag = pcg(mu, dx, r, pv, z, prm.eps_c, prm.maxiter_pcg, &pcg_i);   // :375
      pcg_total += pcg_i;
      if (pcg_flag > 0) { flag = 2; break; }                            // :377-381
      double ar_dot = -dot(gv, dx, N);
      double alpha = 1.0, s = 0;
      for (int k = g.lane; k < N; k += G::SIZE) {                       // :384-391
        double xk = xnew[k]; pv[k] = xk;
        xk -= alpha * dx[k]; xnew[k] = xk;
        double t = xk - xtil[k]; gv[k] = t; s += t * t;
      }
      double dist2 = g.sum(s);
      g.sync();
      c_aux(cval, xnew);                                                // :392
      if (ineq) calculate_h(cvaug, xnew);
      for (int a = g.lane; a < ME; a += G::SIZE) cvaug[M - ME + a] = cval[a];
      g.sync();
      int armijo_count = 0;
      while (dot(cvaug, cvaug, M) + mu * dist2 > prev_obj + 1e-4 * alpha * ar_dot) {   // :403
        alpha /= 2; s = 0;
        for (int k = g.lane; k < N; k += G::SIZE) {
          double xk = pv[k] - alpha * dx[k]; xnew[k] = xk;
          double t = xk - xtil[k]; gv[k] = t; s += t * t;
        }
        dist2 = g.sum(s);
        g.sync();
        // :410-417 -- the reference evaluates c! into cvalaug and then overwrites it with the stale cval of the
        // alpha=1 trial, so the c-part of the merit is frozen; only the bound part h is refreshed.
        if (ineq) calculate_h(cvaug, xnew);
        armijo_count++; st.pp_backtracks++;
        if (armijo_count == 100) { flag = 3; break; }
      }
      i++;
      mu = fmin(mu * 0.1, sqrt(dot(cvaug, cvaug, M)));                  // :431
    }
    if (i == prm.maxiter_retract) flag = 1;
    *it1 = i; *it2 = pcg_total;
    return flag;
  }

  // ------------------------------------------------------------ retract!(::NR) (retractions.jl:75-177), Cholesky-QR basis
  LFPSQP_DEV void nr_apply_basis(const double *delta) {  // xnew += Q delta, Q = PJct L^-T
    for (int a = g.lane; a < ME; a += G::SIZE) ub[a] = delta[a];
    g.sync();
    solveLt(ub);
    for (int j = g.lane; j < NA; j += G::SIZE) {
      double wj = coldot(ub, j);
      if (ineq) { double dx = Dx[j], dy = Dy[j]; xnew[j] += dy * dy * wj; xnew[NA + j] -= dx * dy * wj; }
      else xnew[j] += wj;
    }
    g.sync();
  }
  LFPSQP_DEV int retract_nr(int *it1) {
    double *t1 = nrt, *t2 = nrt + ME, *dc = nrt + 2 * ME;
    copy(xnew, xtil, N);
    if (ineq) y_retract(xnew, x);
    c_aux(cval, xnew);
    // D0 = L^-1 (replaces Sigma^-1 V', :126-130): column c of L^-1 by forward substitution, one column per lane
    for (int c = g.lane; c < ME; c += G::SIZE) {
      for (int i = 0; i < ME; i++) {
        double s = (i == c) ? 1.0 : 0.0;
        for (int t = c; t < i; t++) s -= Gm[i * ME + t] * Dnr[t * ME + c];
        Dnr[i * ME + c] = (i < c) ? 0.0 : s / Gm[i * ME + i];
      }
    }
    g.sync();
    int i = 0;
    while (i < prm.maxiter_retract) {
      if (norminf(cval, ME) < prm.eps_c) break;
      for (int a = g.lane; a < ME; a += G::SIZE) {           // :140 delta = -D c
        double s = 0; for (int b = 0; b < ME; b++) s += Dnr[a * ME + b] * cval[b];
        t1[a] = -s;
      }
      g.sync();
      nr_apply_basis(t1);                                    // :141
      if (ineq) y_retract(xnew, x);
      c_aux(t2, xnew);
      for (int a = g.lane; a < ME; a += G::SIZE) { dc[a] = t2[a] - cval[a]; cval[a] = t2[a]; }
      g.sync();
      for (int a = g.lane; a < ME; a += G::SIZE) {           // :156 t2 = D' delta
        double s = 0; for (int b = 0; b < ME; b++) s += Dnr[b * ME + a] * t1[b];
        t2[a] = s;
      }
      g.sync();
      double den = dot(t2, dc, ME);
      for (int a = g.lane; a < ME; a += G::SIZE) {           // :157 t1 = delta - D dc
        double s = 0; for (int b = 0; b < ME; b++) s += Dnr[a * ME + b] * dc[b];
        t1[a] -= s;
      }
      g.sync();
      double al = 1.0 / den;
      for (int e = g.lane; e < ME * ME; e += G::SIZE) Dnr[e] += al * t1[e / ME] * t2[e % ME];   // ger! :160
      g.sync();
      i++;
    }
    *it1 = i;
    return (i == prm.maxiter_retract) ? 1 : 0;
  }

  // kind: 0 Euclidean, 1 YRetract, 2 NR, 3 ProjPenalty (optimize.jl:396-412)
  LFPSQP_DEV int retract(int kind, int *it1, int *it2) {
    *it1 = 0; *it2 = 0;
    int flag = 0;
    if (kind == 0) copy(xnew, xtil, N);
    else if (kind == 1) { copy(xnew, xtil, N); y_retract(xnew, x); }
    else if (kind == 2) flag = retract_nr(it1);
    else flag = retract_pp(it1, it2);
    st.retract_outer += *it1; st.retract_pcg += *it2;
    return flag;
  }

  // ------------------------------------------------------------ armijo! (linesearch.jl:32-89)
  LFPSQP_DEV int armijo(int kind, double fval, double *newf_o, double *f_diff_o, double *step_diff_o) {
    double f_diff = INFINITY, step_diff = INFINITY, alpha = prm.alpha, newf = 0.0;
    int flag = 0;
    double ar_dot = dot(d, gr, N);
    ls_it1 = ls_it2 = 0;
    while (step_diff > prm.eps_x) {
      for (int k = g.lane; k < N; k += G::SIZE) xtil[k] = x[k] + alpha * d[k];
      g.sync();
      int i1, i2;
      flag = retract(kind, &i1, &i2);
      ls_it1 += i1; ls_it2 += i2;
      st.armijo_trials++;
      // linesearch.jl:57-60 has no lower bound on alpha in this branch: when the retraction fails at EVERY alpha the
      // reference spins forever once alpha has underflowed to 0.  Stop at the floor the other branch uses (:82-85):
        // flag 98, LFPSQP_ST_NONFINITE.
      if (flag > 0) { if (alpha < 1e-100) { flag = 98; break; } alpha *= prm.s; continue; }   // :57-60
      newf = f_aux(xnew);
      double s = 0;
      for (int k = g.lane; k < NA; k += G::SIZE) { double t = xnew[k] - x[k]; s += t * t; }   // :66 first n entries
      step_diff = sqrt(g.sum(s));
      f_diff = fabs(newf - fval);
      if (prm.disable_linesearch) break;
      if ((newf - fval) <= prm.sigma * alpha * ar_dot) break;             // :75
      alpha *= prm.s;
      if (alpha < 1e-100) { flag = 99; break; }                           // :82-85
    }
    *newf_o = newf; *f_diff_o = f_diff; *step_diff_o = step_diff;
    ls_alpha = alpha;
    return flag;
  }

  // ------------------------------------------------------------ exact_linesearch! (linesearch.jl:107-339)
  // golden-section search with bracketing; every trial point is retracted.  Four rotating point buffers.
  LFPSQP_DEV int exact_linesearch(int kind, double fval, double *newf_o, double *f_diff_o, double *step_diff_o) {
    const double phi1 = (3.0 - sqrt(5.0)) / 2.0, phi2 = (sqrt(5.0) - 1.0) / 2.0, phi3 = (sqrt(5.0) + 1.0) / 2.0;
    double Delta = prm.alpha;
    double f_a = 0, f_b = 0, f_c = 0, f_d = 0, a_a = 0, a_b = 0, a_c = 0, a_d = 0;
    double *x_a = sm + L.o_ex[0], *x_b = sm + L.o_ex[1], *x_c = sm + L.o_ex[2], *x_d = sm + L.o_ex[3], *swp;
    bool do_shrinking = true;
    int flag = 0, i1, i2;
    // trial point pt = x + al*d, retracted in place
    auto TRIAL = [&](double *pt, double al) {
      for (int k = g.lane; k < N; k += G::SIZE) xtil[k] = x[k] + al * d[k];
      g.sync();
      flag = retract(kind, &i1, &i2);
      ls_it1 += i1; ls_it2 += i2;
      st.armijo_trials++;
      copy(pt, xnew, N);
    };
    ls_it1 = ls_it2 = 0;
    copy(x_d, x, N); f_d = fval;
    while (true) {                                             // growing (:150-189)
      swp = x_b; x_b = x_c; x_c = x_d; x_d = swp;
      f_b = f_c; f_c = f_d; a_b = a_c; a_c = a_d;
      TRIAL(x_d, a_d + Delta);
      a_d += Delta;
      if (flag > 0 || a_d > 1.0) { f_d = INFINITY; break; }
      f_d = f_aux(x_d);
      if (f_d > f_c) break;
      do_shrinking = false;
      Delta *= phi3;
    }
    if (do_shrinking) {                                        // (:192-239)
      f_b = fval; a_b = 0.0; copy(x_b, x, N);
      f_c = INFINITY; a_c = Delta;
      swp = x_d; x_d = x_c; x_c = swp;
      while (true) {
        swp = x_d; x_d = x_c; x_c = swp;
        f_d = f_c; a_d = a_c;
        TRIAL(x_c, phi1 * a_c);
        a_c *= phi1;
        if (flag > 0 || a_c > 1.0) f_c = INFINITY; else f_c = f_aux(x_c);
        if (f_c <= fval || a_c < 1e-100) break;
      }
    }
    f_a = f_b; f_b = f_c; a_a = a_b; a_b = a_c;                // (:242-266)
    swp = x_a; x_a = x_b; x_b = x_c; x_c = swp;
    a_c = a_a + phi2 * (a_d - a_a);
    TRIAL(x_c, a_c);
    if (flag > 0 || a_c > 1.0) f_c = INFINITY; else f_c = f_aux(x_c);
    const double nd_ = sqrt(dot(d, d, N));
    while ((a_c - a_b) > 1e-6 * nd_) {                         // golden-section main loop (:270-322)
      if (f_b < f_c || isinf(f_c)) {
        swp = x_d; x_d = x_c; x_c = x_b; x_b = swp;
        f_d = f_c; f_c = f_b; a_d = a_c; a_c = a_b;
        a_b = a_a + phi1 * (a_d - a_a);
        TRIAL(x_b, a_b);
        f_b = f_aux(x_b);
      } else {
        swp = x_a; x_a = x_b; x_b = x_c; x_c = swp;
        f_a = f_b; f_b = f_c; a_a = a_b; a_b = a_c;
        a_c = a_a + phi2 * (a_d - a_a);
        TRIAL(x_c, a_c);
        if (flag > 0 || a_c > 1.0) f_c = INFINITY; else f_c = f_aux(x_c);
      }
    }
    (void)f_a; (void)f_d;
    double newf;
    if (f_b < f_c) { copy(xnew, x_b, N); newf = f_b; ls_alpha = a_b; } else { copy(xnew, x_c, N); newf = f_c; ls_alpha = a_c; }   // (:325-333)
    double s = 0;
    for (int k = g.lane; k < NA; k += G::SIZE) { double t = xnew[k] - x[k]; s += t * t; }
    *step_diff_o = sqrt(g.sum(s));
    *f_diff_o = fabs(newf - fval);
    *newf_o = newf;
    return flag;
  }

  // ------------------------------------------------------------ the driver (optimize.jl:176-443)
  LFPSQP_DEV void run(const BatchedArgs &A, int64_t k) {
    fc.prm = A.fam_params ? A.fam_params + k * A.fam_stride : nullptr;
    if constexpr (Fam::kId == LFPSQP_FAM_QCQP) { fc.k = k; fc.qp = A.qcqp; }
    st = lfpsqp_stats{}; status = 0;
    for (int i = g.lane; i < L.total; i += G::SIZE) sm[i] = 0.0;
    g.sync();
    for (int i = g.lane; i < n; i += G::SIZE) x[i] = A.x0[k * n + i];
    g.sync();
    if (p > 0) {  // slack start values s0 = d(x0) (optimize.jl:26-28)
      Fam::d(g, fc, x + n, x);
      g.sync();
    }
    if (ineq) generate_initial_y(x);                                       // :180-182
    int64_t it = 0;
    double f_diff = INFINITY, step_diff = INFINITY, kkt_diff = INFINITY, prev_grad_norm = 0.0;
    double fval = f_aux(x);                                                // :249-250
    int64_t nobj = 0;
    if (g.lane == 0 && nobj < A.H) A.obj_hist[k * A.H + nobj] = fval;
    nobj++;
    if (ME > 0) c_aux(cval, x);                                            // :252
    int cond = LFPSQP_F_TOL;
    while (true) {
      grad_aux(gr, x);                                                     // :259
      for (int i = g.lane; i < N; i += G::SIZE) d[i] = -1.0 * gr[i];       // :262
      if (A.noise) {                                                       // :264-273, caller-supplied noise rows
        const double nc = noise_coef(prm, it, A.noise_T);
        if (nc != 0.0) { const double *nz = A.noise + ((int64_t)k * A.noise_T + it) * N; for (int i = g.lane; i < N; i += G::SIZE) d[i] += nc * nz[i]; }
      }
      g.sync();
      if (ineq) inequality_gradient(x);                                    // :277
      if (ME > 0) {
        jac_aux(cval, x);                                                  // :283
        factor();
        if (pinv) status |= LFPSQP_ST_RANK_DEFICIENT;   // informational: the truncated path of optimize.jl:297-302 was taken
      }
      project(d, true);                                                    // :306-307 / :316-317 + multipliers :331-343
      kkt_diff = norminf(d, N);                                            // :320
      if (f_diff <= prm.eps_f) { cond = LFPSQP_F_TOL; break; }             // :347-359
      else if (step_diff <= prm.eps_x) { cond = LFPSQP_X_TOL; break; }
      else if (it >= prm.maxiter) { cond = LFPSQP_MAX_ITER; break; }
      else if (kkt_diff <= prm.eps_kkt) { cond = LFPSQP_KKT_TOL; break; }
      if (!(kkt_diff == kkt_diff)) { status |= LFPSQP_ST_NONFINITE; cond = LFPSQP_MAX_ITER; break; }
      if (prm.do_newton) {                                                 // :364-390
        double gn = sqrt(dot(d, d, N));
        double tol = prm.tn_kappa * fmin(1.0, gn / prev_grad_norm) * gn;
        prev_grad_norm = gn;
        double tn_res;
        projcg(d, ineq ? NA + rank : rank, tol, prm.tn_maxiter, &tn_res);        // c has length rank / n+rank (:366-372)
        if (dot(nd, d, N) > 0.0) { copy(d, nd, N); st.newton_accepted++; }
      }
      int kind;                                                            // :396-412
      if (ME > 0) kind = (rank == ME && !prm.do_project_retract) ? 2 : 3;
      else kind = ineq ? 1 : 0;
      double newf;
      int flag;                                                            // :415-420
      if (prm.linesearch == 0 || prm.disable_linesearch) flag = armijo(kind, fval, &newf, &f_diff, &step_diff);
      else flag = exact_linesearch(kind, fval, &newf, &f_diff, &step_diff);
      st.flag_last = flag;
      if (flag == 98) { status |= LFPSQP_ST_NONFINITE; cond = LFPSQP_MAX_ITER; break; }
      copy(x, xnew, N);                                                    // :424-426
      fval = newf;
      if (g.lane == 0 && nobj < A.H) A.obj_hist[k * A.H + nobj] = fval;
      nobj++;
      it++;
    }
    for (int i = g.lane; i < n; i += G::SIZE) A.x_out[k * n + i] = x[i];   // :442 (x[1:n] of the user problem, :68)
    for (int a = g.lane; a < ME; a += G::SIZE) A.lambda[k * ME + a] = lam[a];
    if (g.lane == 0) {
      A.obj_len[k] = nobj;
      lfpsqp_term t; t.condition = cond; t.status = status; t.f_diff = f_diff; t.step_diff = step_diff;
      t.kkt_diff = kkt_diff; t.iter = it;
      A.term[k] = t;
      if (A.stats) A.stats[k] = st;
    }
  }
};

// Persistent CTAs; every warp pulls instance indices from a global counter until the batch is drained
// (absorbs the per-instance iteration-count variance).
template <class Fam>
__global__ void __launch_bounds__(256, 2) batched_warp_kernel(const BatchedArgs A, const int use_nr) {
  extern __shared__ double smem[];
  const WarpLayout L(A.n, A.m, A.p, A.ineq, use_nr, (A.prm.linesearch != 0 && !A.prm.disable_linesearch) ? 1 : 0);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  // CTA-shared copy of the bound data
  double *bnd = smem;
  const int nb = A.ineq ? 5 * L.NA : 0;
  for (int i = threadIdx.x; i < nb; i += blockDim.x) bnd[i] = A.bnd[i];
  __syncthreads();
  double *ws = smem + ((nb + 1) & ~1) + (size_t)warp * L.total;
  (void)nwarps;
  WarpGroup g(lane);
  Solver<Fam, WarpGroup> S(g, L, A.prm, ws, bnd);
  for (;;) {
    unsigned long long k = 0;
    if (lane == 0) k = atomicAdd(A.work_counter, 1ULL);
    k = __shfl_sync(0xffffffffu, k, 0);
    if ((int64_t)k >= A.B) break;
    S.run(A, (int64_t)k);
  }
}

}  // namespace lfpsqp
