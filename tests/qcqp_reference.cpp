/*
 * tests/qcqp_reference.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * The dense QCQP family (LFPSQP_FAM_QCQP) for the CPU oracle.  The oracle's source is compiled into this library
 * unchanged -- the same driver, the same dot / gemv helpers and g_flops accounting, the same three builds (plain, FMA,
 * left-to-right summation; tests/qcqp_reference.py) -- and this file adds one family beside the registered ones.
 * qorc_* are the oracle's optimize / optimize_batched / family_* entry points with the family table extended by
 * ORC_FAM_QCQP; every other family id resolves exactly as in the oracle.
 */
#define make_family make_family_registered
#include "../oracle/lfpsqp_oracle.cpp"
#undef make_family

enum { ORC_FAM_QCQP = 101 };

/* dense QCQP: f = 1/2 x'Px + q.x + r, c_i = 1/2 x'Qc_i x + Ac_i.x - bc_i, d_k likewise (matrices symmetric);
   params = [P(n*n) | q(n) | r | Qc(m*n*n) | Ac(m*n) | bc(m) | Qd(p*n*n) | Ad(p*n) | bd(p)], zero where an array is absent.
   A quadratic's value is dot(0.5 Mx + a, x) and its gradient Mx + a: with the README families' encodings every extra
   term is an exact zero or an exact power-of-two scaling, so they reproduce the registered families bit for bit. */
struct Qcqp : Family {
  const double *P, *q, *r, *Qc, *Ac, *bc, *Qd, *Ad, *bd;
  vec u, w;
  Qcqp(int64_t n_, int64_t m_, int64_t p_, const double *prm) : u(n_), w(n_) {
    n = n_; m = m_; p = p_;
    P = prm; q = P + n * n; r = q + n; Qc = r + 1; Ac = Qc + m * n * n; bc = Ac + m * n; Qd = bc + m; Ad = Qd + p * n * n;
    bd = Ad + p * n;
  }
  /* 1/2 x'Mx + a.x; writes the gradient Mx + a to row[j * ld] when row != NULL */
  double quad(const double *M, const double *a, const double *x, double *row, int64_t ld) {
    gemv('N', n, n, 1.0, M, n, x, 0.0, u.data());
    for (int64_t j = 0; j < n; j++) { if (row) row[j * ld] = u[j] + a[j]; w[j] = 0.5 * u[j] + a[j]; }
    g_flops += 4.0 * n;
    return dot(w.data(), x, n);
  }
  double f(const double *x) override { return quad(P, q, x, nullptr, 0) + r[0]; }
  void grad(double *g, const double *x) override {
    gemv('N', n, n, 1.0, P, n, x, 0.0, g);
    for (int64_t j = 0; j < n; j++) g[j] += q[j];
    g_flops += (double)n;
  }
  void c(double *cv, const double *x) override {
    for (int64_t i = 0; i < m; i++) cv[i] = quad(Qc + i * n * n, Ac + i * n, x, nullptr, 0) - bc[i];
  }
  void jac(double *J, int64_t ld, double *cv, const double *x) override {
    for (int64_t i = 0; i < m; i++) cv[i] = quad(Qc + i * n * n, Ac + i * n, x, J + i, ld) - bc[i];
  }
  void d(double *dv, const double *x) override {
    for (int64_t k = 0; k < p; k++) dv[k] = quad(Qd + k * n * n, Ad + k * n, x, nullptr, 0) - bd[k];
  }
  void jacd(double *J, int64_t ld, double *dv, const double *x) override {
    for (int64_t k = 0; k < p; k++) dv[k] = quad(Qd + k * n * n, Ad + k * n, x, J + k, ld) - bd[k];
  }
  void hess(double *dest, const double *v, const double *, const double *lam, const double *lam_d) override {
    gemv('N', n, n, 1.0, P, n, v, 0.0, dest);
    for (int64_t i = 0; i < m; i++) gemv('N', n, n, lam[i], Qc + i * n * n, n, v, 1.0, dest);
    for (int64_t k = 0; k < p; k++) gemv('N', n, n, lam_d[k], Qd + k * n * n, n, v, 1.0, dest);
  }
};

static std::unique_ptr<Family> make_family(int family, const double *prm, int64_t n, int64_t m, int64_t p) {
  if (family == ORC_FAM_QCQP) return std::unique_ptr<Family>(new Qcqp(n, m, p, prm));
  return make_family_registered(family, prm, n, m, p);
}

/* ---- orc_optimize / orc_optimize_batched / orc_family_* with the extended family table ---- */
extern "C" int qorc_optimize(int family, const double *fam_params, int64_t n, int64_t m, int64_t p, const double *x0,
                             const double *xl, const double *xu, const orc_params *prm, double *x_out, double *obj_hist,
                             int64_t obj_cap, int64_t *obj_len, double *lambda, orc_term *term, orc_stats *stats) {
  auto F = make_family(family, fam_params, n, m, p);
  if (!F) return -1;
  orc_stats local; memset(&local, 0, sizeof(local));
  g_stats = &local; g_flops = 0.0;
  int rc;
  if (p == 0) {                                                 /* optimize.jl:15-17 -> :88-104 */
    PlainProblem P(*F);
    rc = core(P, x0, xl, xu, *prm, x_out, obj_hist, obj_cap, obj_len, lambda, term);
  } else {                                                      /* optimize.jl:13-71 via :83-85 (dl=-Inf, du=0) */
    SlackProblem P(*F);
    vec x0a(n + p), xla(n + p), xua(n + p), xo(n + p);
    std::copy(x0, x0 + n, x0a.begin());
    F->d(x0a.data() + n, x0);                                   /* :28 */
    for (int64_t i = 0; i < n; i++) { xla[i] = xl ? xl[i] : -INF; xua[i] = xu ? xu[i] : INF; }
    for (int64_t k = 0; k < p; k++) { xla[n + k] = -INF; xua[n + k] = 0.0; }
    rc = core(P, x0a.data(), xla.data(), xua.data(), *prm, xo.data(), obj_hist, obj_cap, obj_len, lambda, term);
    if (rc == 0) std::copy(xo.begin(), xo.begin() + n, x_out);  /* :68 */
  }
  local.flops = g_flops;
  if (stats) *stats = local;
  g_stats = nullptr;
  return rc;
}

extern "C" int qorc_optimize_batched(int family, const double *fam_params, int64_t fam_stride, int64_t n, int64_t m,
                                     int64_t p, int64_t B, const double *x0, const double *xl, const double *xu,
                                     const orc_params *prm, double *x_out, double *obj_hist, int64_t H, int64_t *obj_len,
                                     double *lambda, orc_term *term, orc_stats *stats, int nthreads) {
  if (nthreads < 1) nthreads = 1;
  std::atomic<int64_t> next(0); std::atomic<int> err(0);
  auto worker = [&]() {
    for (;;) {
      int64_t k0 = next.fetch_add(64);
      if (k0 >= B) break;
      for (int64_t k = k0; k < std::min(B, k0 + 64); k++) {
        t_noise = g_noise ? g_noise + k * g_noise_stride : nullptr;
        int rc = qorc_optimize(family, fam_params ? fam_params + k * fam_stride : nullptr, n, m, p, x0 + k * n, xl, xu,
                               prm, x_out + k * n, obj_hist + k * H, H, obj_len + k, lambda + k * (m + p), term + k,
                               stats ? stats + k : nullptr);
        if (rc) err = rc;
      }
    }
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nthreads; t++) th.emplace_back(worker);
  worker();
  for (auto &t : th) t.join();
  return err;
}

extern "C" double qorc_family_f(int family, const double *prm, int64_t n, int64_t m, int64_t p, const double *x) {
  auto F = make_family(family, prm, n, m, p); return F ? F->f(x) : QNAN;
}
extern "C" void qorc_family_grad(int family, const double *prm, int64_t n, int64_t m, int64_t p, const double *x, double *g) {
  auto F = make_family(family, prm, n, m, p); if (F) F->grad(g, x);
}
extern "C" void qorc_family_jac(int family, const double *prm, int64_t n, int64_t m, int64_t p, const double *x, double *Jc,
                                double *cval) {
  auto F = make_family(family, prm, n, m, p); if (!F) return;
  int64_t M = m + p;
  for (int64_t k = 0; k < M * n; k++) Jc[k] = 0;
  if (m) F->jac(Jc, M, cval, x);
  if (p) F->jacd(Jc + m, M, cval + m, x);
}
extern "C" void qorc_family_hess(int family, const double *prm, int64_t n, int64_t m, int64_t p, const double *x,
                                 const double *lam, const double *src, double *dest) {
  auto F = make_family(family, prm, n, m, p); if (F) F->hess(dest, src, x, lam, lam + m);
}
