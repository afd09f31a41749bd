// batched_reg.cuh -- register-resident solver for SEPARABLE families (BASELINE config C2): one lane GROUP per instance.
//
// Same algorithm, same reference line mapping as batched_warp.cuh (the shared-memory solver), but the vectors of the hot
// loops live in REGISTERS: a group of LW lanes (LW = 32, 16 or 8: 1, 2 or 4 instances per warp) owns one instance; element
// j of an N_A-vector sits in lane j%LW of the group, slot j/LW (NPL slots per lane); the x- and y-halves of the
// 2n-embedding (src/inequality_helper.jl) are two register arrays.  Elementwise work needs no synchronisation at all;
// the only cross-lane traffic is the xor-butterfly of the dot products (log2 LW stages, group-masked shuffles).  The
// m_E (<= 2) rows of J, the m_E x m_E Gram/Cholesky factor and all m_E-vectors are replicated in registers of every lane.
//
// Why groups narrower than a warp: the kernel is bound by FP64 issue and by the latency of dependent shuffle / division
// chains, not by memory.  Every per-instance SCALAR operation (CG coefficients, divisions, square roots, the Cholesky of
// the m_E x m_E Gram) costs one warp instruction whatever the group width, and every reduction costs log2(LW) shuffle
// stages: with 2 (4) instances per warp these costs are shared by 2 (4) instances, the butterflies lose one (two) stages,
// and every lane carries 2x (4x) the independent elementwise work (ILP) that hides the FP64 latency.  Instances of one
// warp run the five-deep data-dependent loop nest under the hardware's divergence handling (group-masked shuffles);
// the groups of a warp re-converge at every loop exit, so the cost is the max of the trip counts (BASELINE C2: the
// per-instance counts are identical for 93 % of the instances and differ by one projcg iteration for the rest).
//
// Vectors that are cold during a hot loop (the iterate x and the direction d during the retraction, xtilde / xnew / the
// right-hand side during pcg!) are parked in a group-private shared-memory stash (each lane reads back exactly the
// elements it wrote: no synchronisation), which keeps the kernel at <= 168 registers (12 warps/SM) without spills.
//
// "Separable" = f(x) = sum_j f_j(x_j), every constraint c_a(x) = sum_j c_aj(x_j) - off_a, hence a diagonal Lagrangian
// Hessian: README equality / inequality examples (README.md:41-76), the bounded quadratic, diagonal-quadratic rows.
// Anything else (Thomson, Rosenbrock, sin system, m_E > 2, n_A > 128) runs in batched_warp.cuh.
#pragma once
#include "common.cuh"

// Alternatives measured against this kernel on a B200 (C2, LW = 8: 1.687 ms for 65,536 instances) and dropped: bit masks
// for "slot holds a user variable / a slack" instead of index compares 1.82 ms; the line formula for every slot plus one
// fix-up branch per lane 1.76 ms; pcg!'s dx accumulated in the stash 2.04 ms; family parameters re-read through the L1
// instead of cached in registers 1.72 ms (profiles/r2_c2_ab_feature_switches.log).  With the line head (HEAD = NPL - 1,
// 1.389 ms): user-variable and line-gradient facts made compile-time in the head slots as well 1.288 ms, but the
// constants change how the compiler contracts those slots' expressions into FMAs (results differ in the last bits);
// the head at 168 registers (MINB = 3) spills 1.4 KB and is slower, 1.76 ms (profiles/r3_c2_line_head_ab.log).

namespace lfpsqp {

// ---------------------------------------------------------------- separable family descriptions
// row a < m is an equality c_a, row a >= m an inequality d_{a-m}; ep = this element's cached parameters (KP doubles)
struct SepReadmeIneq {  // f = coeff.x ; d = x.x - 1     (README.md:57-76)
  static constexpr int kId = LFPSQP_FAM_README_INEQ, KP = 1;
  static LFPSQP_DEV void load(const FamCtx &fc, int j, double *ep) { ep[0] = __ldg(fc.prm + j); }
  static LFPSQP_DEV double f(const FamCtx &, int, double x, const double *ep) { return ep[0] * x; }
  static LFPSQP_DEV double g(const FamCtx &, int, double, const double *ep) { return ep[0]; }
  static LFPSQP_DEV double h(const FamCtx &, int, double, const double *, const double *lam) { return 2.0 * lam[0]; }
  static LFPSQP_DEV double c(const FamCtx &, int, int, double x, const double *) { return x * x; }
  static LFPSQP_DEV double off(const FamCtx &, int) { return 1.0; }
  static LFPSQP_DEV double jac(const FamCtx &, int, int, double x, const double *) { return 2.0 * x; }
};
struct SepReadmeEq {  // f = x.x ; c = x[1] - 0.75          (README.md:41-54)
  static constexpr int kId = LFPSQP_FAM_README_EQ, KP = 0;
  static LFPSQP_DEV void load(const FamCtx &, int, double *) {}
  static LFPSQP_DEV double f(const FamCtx &, int, double x, const double *) { return x * x; }
  static LFPSQP_DEV double g(const FamCtx &, int, double x, const double *) { return 2.0 * x; }
  static LFPSQP_DEV double h(const FamCtx &, int, double, const double *, const double *) { return 2.0; }
  static LFPSQP_DEV double c(const FamCtx &, int, int j, double x, const double *) { return j == 0 ? x : 0.0; }
  static LFPSQP_DEV double off(const FamCtx &, int) { return 0.75; }
  static LFPSQP_DEV double jac(const FamCtx &, int, int j, double, const double *) { return j == 0 ? 1.0 : 0.0; }
};
struct SepBoxQuad {  // f = |x-t|^2 ; optional c = a.x - b ; params [t(n), a(n), b]
  static constexpr int kId = LFPSQP_FAM_BOXQUAD, KP = 2;
  static LFPSQP_DEV void load(const FamCtx &fc, int j, double *ep) { ep[0] = __ldg(fc.prm + j); ep[1] = __ldg(fc.prm + fc.n + j); }
  static LFPSQP_DEV double f(const FamCtx &, int, double x, const double *ep) { double u = x - ep[0]; return u * u; }
  static LFPSQP_DEV double g(const FamCtx &, int, double x, const double *ep) { return 2.0 * (x - ep[0]); }
  static LFPSQP_DEV double h(const FamCtx &, int, double, const double *, const double *) { return 2.0; }
  static LFPSQP_DEV double c(const FamCtx &, int, int, double x, const double *ep) { return ep[1] * x; }
  static LFPSQP_DEV double off(const FamCtx &fc, int) { return __ldg(fc.prm + 2 * fc.n); }
  static LFPSQP_DEV double jac(const FamCtx &, int, int, double, const double *ep) { return ep[1]; }
};


#define LF_UNROLL _Pragma("unroll")

// NaN-propagating max of two values that are >= 0 or NaN with a clear sign bit (every use takes fabs first): for such
// doubles the IEEE order is the integer order of the bit patterns and every NaN sorts above +Inf, so an integer max
// returns what pmax returns, on the integer pipe instead of two FP64 compares.
LFPSQP_DEV double pmax_nn(double a, double b) {
  const long long ia = __double_as_longlong(a), ib = __double_as_longlong(b);
  return __longlong_as_double(ia > ib ? ia : ib);
}

// xor-butterflies over a group of LW lanes (every lane of the group ends with the bitwise-identical result)
template <int LW> LFPSQP_DEV double gsum(unsigned mask, double v) {
  LF_UNROLL for (int o = LW / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
  return v;
}
template <int LW> LFPSQP_DEV double gmax(unsigned mask, double v) {
  LF_UNROLL for (int o = LW / 2; o > 0; o >>= 1) v = pmax_nn(v, __shfl_xor_sync(mask, v, o));
  return v;
}
// independent butterflies interleaved (same instruction count, one dependent-latency chain instead of two / three)
template <int LW> LFPSQP_DEV void gsum2(unsigned mask, double &a, double &b) {
  LF_UNROLL for (int o = LW / 2; o > 0; o >>= 1) {
    double ta = __shfl_xor_sync(mask, a, o), tb = __shfl_xor_sync(mask, b, o);
    a += ta; b += tb;
  }
}
template <int LW> LFPSQP_DEV void gsum3(unsigned mask, double &a, double &b, double &c) {
  LF_UNROLL for (int o = LW / 2; o > 0; o >>= 1) {
    double ta = __shfl_xor_sync(mask, a, o), tb = __shfl_xor_sync(mask, b, o), tc = __shfl_xor_sync(mask, c, o);
    a += ta; b += tb; c += tc;
  }
}
template <int LW> LFPSQP_DEV void gmax_sum2(unsigned mask, double &mx, double &a, double &b) {
  LF_UNROLL for (int o = LW / 2; o > 0; o >>= 1) {
    double tm = __shfl_xor_sync(mask, mx, o), ta = __shfl_xor_sync(mask, a, o), tb = __shfl_xor_sync(mask, b, o);
    mx = pmax_nn(mx, tm); a += ta; b += tb;
  }
}

// HEAD: slots 0 .. HEAD-1 of every lane hold only line pairs (bound kind 0, q = r = s = t = 0; checked by the
// launcher).  There the bound kind and the bound table are compile-time, so calculate_h is x - y, inequality_gradient,
// y_retract_elem and generate_initial_y take the line branch, and the parabola / circle code and the table reads are not
// emitted.  The line gradients and the user / slack tests stay runtime values in every slot: that keeps every
// expression compiled as with HEAD = 0 (same FMA contraction, bitwise-identical results).
template <class Fam, int LW, int NPL, int ME, bool INEQ, bool SPARSE, int HEAD>
struct RegSolver {
  static constexpr int KP = Fam::KP > 0 ? Fam::KP : 1;
  static constexpr int MEA = ME > 0 ? ME : 1;
  static constexpr int NAP = NPL * LW;                       // padded vector length (bound tables are zero-padded to it)
  static constexpr int VECD = (INEQ ? 2 : 1) * NAP;          // doubles of one stashed vector
  static constexpr int NGR = SPARSE ? 1 : NPL;
  enum { SV_X = 0, SV_D, SV_XTIL, SV_XNEW, SV_GV, SV_COUNT };
  static constexpr int STASH_DOUBLES = SV_COUNT * VECD;      // per group
  static constexpr int GPW = 32 / LW;                        // groups per warp
  struct Vec { double x[NPL]; double y[INEQ ? NPL : 1]; };

  const int lane;        // lane within the group
  const unsigned gmask;  // the group's lanes
  const lfpsqp_params &prm;
  FamCtx fc;
  const int n, m, p, NA;
  // bound data (inequality_helper.jl:1-8) in CTA-shared memory: [kind | q | r | s | t] x NAP, zero beyond N_A
  // (kind: 0 line, 1 parabola, 2 circle); padded elements have q = s = r = t = 0 and x = y = 0 throughout
  const double *bnd;
  unsigned kinds;        // 2 bits per slot: this lane's bound kinds (bkind without the shared-memory read)
  double pcg_rho_stop;   // largest rho with sqrt(rho) <= eps_c: pcg!'s test norm(r) > tol (retractions.jl:207) without the sqrt
  double *stash;         // this lane's first element in its warp's parking area (see sx)
  double ep[NPL][KP];    // cached per-element family parameters
  // instance state
  Vec x;
  double J[MEA][NPL], Lc[MEA][MEA], cval[MEA], lam[MEA];
  // inequality_gradient! output.  SPARSE (every lane holds at most ONE pair that is not a line; checked by the launcher):
  // line pairs carry the constants S = sqrt(2), Dx = 1/S, Dy = -1/S (see inequality_gradient), so only the exceptional
  // slot `exc` (-1: none) of the lane is stored -- 3 doubles instead of 3 NPL
  double Dx[NGR], Dy[NGR], S[NGR], lamy[NPL];
  int exc;
  double cvh[NPL], cvc[MEA];   // cvalaug = [h ; c] (retractions.jl:29), persistent across PP calls (stale-tail quirk)
  int st_projcg, st_negcurv, st_trials, st_rout, st_rpcg, st_bt, st_newton, st_fact, st_feval, status;
  int rank; bool pinv;   // numerical rank (optimize.jl:297-302); Lc holds the truncated pseudo-inverse G^+ when pinv

  LFPSQP_DEV RegSolver(int lane_, unsigned gmask_, const lfpsqp_params &prm_, int n_, int m_, int p_, const double *bnd_, double *stash_)
      : lane(lane_), gmask(gmask_), prm(prm_), n(n_), m(m_), p(p_), NA(n_ + p_), bnd(bnd_), stash(stash_) {
    fc.n = n_; fc.m = m_; fc.p = p_; fc.prm = nullptr;
    kinds = 0;
    exc = -1;
    if (INEQ) { LF_UNROLL for (int k = 0; k < NPL; k++) { const unsigned kd = (unsigned)(int)bnd[k * LW + lane] & 3u; kinds |= kd << (2 * k); if (kd != 0u) exc = k; } }
    // sqrt is correctly rounded and monotone: {rho : sqrt(rho) <= eps_c} is an interval [0, t]; find t once
    const double e = prm.eps_c;
    if (e < 0.0) pcg_rho_stop = -1.0;
    else if (!(e < INFINITY)) pcg_rho_stop = e;
    else {
      double t = e * e;
      while (t > 0.0 && sqrt(t) > e) t = __longlong_as_double(__double_as_longlong(t) - 1);
      while (sqrt(__longlong_as_double(__double_as_longlong(t) + 1)) <= e) t = __longlong_as_double(__double_as_longlong(t) + 1);
      pcg_rho_stop = t;
    }
  }

  LFPSQP_DEV int idx(int s) const { return s * LW + lane; }
  LFPSQP_DEV bool user(int k) const { return idx(k) < n; }
  LFPSQP_DEV bool slack(int a, int k) const { return a >= m && idx(k) == n + (a - m); }
  LFPSQP_DEV double gS(int k) const { if (!SPARSE) return S[SPARSE ? 0 : k]; return (k == exc) ? S[0] : sqrt(2.0); }
  LFPSQP_DEV double gDx(int k) const { if (!SPARSE) return Dx[SPARSE ? 0 : k]; return (k == exc) ? Dx[0] : 1.0 * (1.0 / sqrt(2.0)); }
  LFPSQP_DEV double gDy(int k) const { if (!SPARSE) return Dy[SPARSE ? 0 : k]; return (k == exc) ? Dy[0] : -1.0 * (1.0 / sqrt(2.0)); }
  LFPSQP_DEV void eload(int k, double *e) const {   // family parameters of user slot k
    LF_UNROLL for (int q = 0; q < KP; q++) e[q] = ep[k][q];
  }
  LFPSQP_DEV int bkind(int k) const { return (INEQ && k >= HEAD) ? (int)((kinds >> (2 * k)) & 3u) : 0; }
  LFPSQP_DEV double bq(int k) const { return (INEQ && k >= HEAD) ? bnd[NAP + idx(k)] : 0.0; }
  LFPSQP_DEV double br(int k) const { return (INEQ && k >= HEAD) ? bnd[2 * NAP + idx(k)] : 0.0; }
  LFPSQP_DEV double bs(int k) const { return (INEQ && k >= HEAD) ? bnd[3 * NAP + idx(k)] : 0.0; }
  LFPSQP_DEV double bt(int k) const { return (INEQ && k >= HEAD) ? bnd[4 * NAP + idx(k)] : 0.0; }
  LFPSQP_DEV double sum(double v) const { return gsum<LW>(gmask, v); }
  LFPSQP_DEV double maxr(double v) const { return gmax<LW>(gmask, v); }
  LFPSQP_DEV void sum2(double &a, double &b) const { gsum2<LW>(gmask, a, b); }
  LFPSQP_DEV void sum3(double &a, double &b, double &c) const { gsum3<LW>(gmask, a, b, c); }

  // ---------------------------------------------------------------- stash (group-private shared memory, lane-private elements)
  // element e = v VECD + idx(k) of a group's area sits at (e - lane) GPW + group_in_warp LW + lane of its warp's area:
  // the groups of a warp are interleaved, so one access by the warp covers 32 consecutive doubles (no bank conflict)
  LFPSQP_DEV double &sx(int v, int k) const { return stash[(v * VECD + k * LW) * GPW]; }
  LFPSQP_DEV double &sy(int v, int k) const { return stash[(v * VECD + NAP + k * LW) * GPW]; }
  LFPSQP_DEV void put(int v, const Vec &a) const {
    LF_UNROLL for (int k = 0; k < NPL; k++) { sx(v, k) = a.x[k]; if (INEQ) sy(v, k) = a.y[k]; }
  }
  LFPSQP_DEV void get(int v, Vec &a) const {
    LF_UNROLL for (int k = 0; k < NPL; k++) { a.x[k] = sx(v, k); if (INEQ) a.y[k] = sy(v, k); }
  }

  // ---------------------------------------------------------------- vector helpers
  LFPSQP_DEV double dot(const Vec &a, const Vec &b) const {
    double s = 0.0;
    LF_UNROLL for (int k = 0; k < NPL; k++) s += a.x[k] * b.x[k];
    if (INEQ) { LF_UNROLL for (int k = 0; k < NPL; k++) s += a.y[k] * b.y[k]; }
    return sum(s);
  }
  LFPSQP_DEV void zero(Vec &a) const {
    LF_UNROLL for (int k = 0; k < NPL; k++) { a.x[k] = 0.0; if (INEQ) a.y[k] = 0.0; }
  }
  // out[a] = sum_j J[a][j] v_j  (J acts on the x-half only)
  LFPSQP_DEV void rowdots(double *out, const double *vx) const {
    if (ME == 2) {
      double s0 = 0.0, s1 = 0.0;
      LF_UNROLL for (int k = 0; k < NPL; k++) { s0 += J[0][k] * vx[k]; s1 += J[MEA - 1][k] * vx[k]; }
      sum2(s0, s1); out[0] = s0; out[MEA - 1] = s1;
      return;
    }
    LF_UNROLL for (int a = 0; a < ME; a++) {
      double s = 0.0;
      LF_UNROLL for (int k = 0; k < NPL; k++) s += J[a][k] * vx[k];
      out[a] = sum(s);
    }
  }
  LFPSQP_DEV double coldot(const double *u, int k) const {
    double s = 0.0;
    LF_UNROLL for (int a = 0; a < ME; a++) s += J[a][k] * u[a];
    return s;
  }
  LFPSQP_DEV void solveG(double *u) const {  // u <- (L L')^-1 u (or G^+ u), replicated scalar code
    if (pinv) {
      double t[MEA];
      LF_UNROLL for (int a = 0; a < ME; a++) { double s = 0.0; LF_UNROLL for (int b = 0; b < ME; b++) s += Lc[a][b] * u[b]; t[a] = s; }
      LF_UNROLL for (int a = 0; a < ME; a++) u[a] = t[a];
      return;
    }
    LF_UNROLL for (int k = 0; k < ME; k++) {
      double s = u[k];
      LF_UNROLL for (int t = 0; t < k; t++) s -= Lc[k][t] * u[t];
      u[k] = s / Lc[k][k];
    }
    LF_UNROLL for (int k = ME - 1; k >= 0; k--) {
      double s = u[k];
      LF_UNROLL for (int t = k + 1; t < ME; t++) s -= Lc[t][k] * u[t];
      u[k] = s / Lc[k][k];
    }
  }

  // ---------------------------------------------------------------- callbacks on the slack-augmented problem (optimize.jl:38-51)
  LFPSQP_DEV double f_aux(const Vec &v) {
    st_feval++;
    double s = 0.0;
    LF_UNROLL for (int k = 0; k < NPL; k++) if (user(k)) { double e[KP]; eload(k, e); s += Fam::f(fc, idx(k), v.x[k], e); }
    return sum(s);
  }
  LFPSQP_DEV void c_partial(double *part, const Vec &v) const {   // un-reduced per-lane partial sums of c_aux
    LF_UNROLL for (int a = 0; a < ME; a++) {
      double s = 0.0;
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        if (user(k)) { double e[KP]; eload(k, e); s += Fam::c(fc, a, idx(k), v.x[k], e); }
        else if (slack(a, k)) s -= v.x[k];               // d_k(x) - s_k
      }
      part[a] = s;
    }
  }
  LFPSQP_DEV void c_aux(double *cv, const Vec &v) const {
    double part[MEA];
    c_partial(part, v);
    if (ME == 2) sum2(part[0], part[MEA - 1]);
    else { LF_UNROLL for (int a = 0; a < ME; a++) part[a] = sum(part[a]); }
    LF_UNROLL for (int a = 0; a < ME; a++) cv[a] = part[a] - Fam::off(fc, a);
  }
  LFPSQP_DEV void jac_fill(const Vec &v) {
    LF_UNROLL for (int a = 0; a < ME; a++)
      LF_UNROLL for (int k = 0; k < NPL; k++)
      {
        double e[KP] = {0.0};
        if (user(k)) eload(k, e);
        J[a][k] = user(k) ? Fam::jac(fc, a, idx(k), v.x[k], e) : ((slack(a, k)) ? -1.0 : 0.0);
      }
  }
  LFPSQP_DEV void jac_aux(double *cv, const Vec &v) {   // jac!(Jc, cval, x): fills J and cval
    jac_fill(v);
    c_aux(cv, v);
  }
  LFPSQP_DEV void hess_aux(Vec &dest, const Vec &src) const {   // Lagrangian Hessian at the current (x, lam, lamy)
    LF_UNROLL for (int k = 0; k < NPL; k++) {
      double e[KP] = {0.0};
      if (user(k)) eload(k, e);
      double hx = user(k) ? Fam::h(fc, idx(k), x.x[k], e, lam) * src.x[k] : 0.0;
      if (INEQ) {
        double ly2 = 2.0 * lamy[k];
        hx += ly2 * bq(k) * src.x[k];
        dest.y[k] = ly2 * bs(k) * src.y[k];
      }
      dest.x[k] = hx;
    }
  }

  // ---------------------------------------------------------------- bound embedding (inequality_helper.jl)
  LFPSQP_DEV void generate_initial_y(Vec &v) const {  // :92-109
    LF_UNROLL for (int k = 0; k < NPL; k++) {
      double xv = v.x[k], yv;
      const int kind = bkind(k);
      if (kind == 0) yv = xv;
      else if (kind == 1) yv = sqrt(fmax(-(xv - bt(k)) / bs(k), 0.0)) + br(k);
      else yv = sqrt(fmax(bt(k) - (xv - br(k)) * (xv - br(k)), 0.0)) + br(k);
      v.y[k] = (idx(k) < NA) ? yv : 0.0;
    }
  }
  LFPSQP_DEV void calculate_h(double *out, const Vec &v) const {  // :112-122
    LF_UNROLL for (int k = 0; k < NPL; k++) {
      // line pairs (and the padded elements) have q = s = r = t = 0: the general formula reduces EXACTLY to x - y there
      if (bkind(k) == 0) { out[k] = v.x[k] - v.y[k]; continue; }
      double q = bq(k), s = bs(k), r = br(k), dx = v.x[k] - r, dy = v.y[k] - r;
      out[k] = q * (dx * dx) + (1.0 - q * q) * v.x[k] + s * (dy * dy) - (1.0 - s * s) * v.y[k] - bt(k);
    }
  }
  LFPSQP_DEV void init_line_gradients() {
    LF_UNROLL for (int k = 0; k < NGR; k++) { const double sv = sqrt(2.0), inv = 1.0 / sv; S[k] = sv; Dx[k] = 1.0 * inv; Dy[k] = -1.0 * inv; }
  }
  LFPSQP_DEV void inequality_gradient(const Vec &v) {  // :125-141
    LF_UNROLL for (int k = 0; k < NPL; k++) {
      if (bkind(k) == 0) { if (!SPARSE) { const double sv = sqrt(2.0), inv = 1.0 / sv; S[SPARSE ? 0 : k] = sv; Dx[SPARSE ? 0 : k] = 1.0 * inv; Dy[SPARSE ? 0 : k] = -1.0 * inv; } continue; }
      double q = bq(k), s = bs(k), r = br(k);
      double dx = 2.0 * q * (v.x[k] - r) + (q == 0.0 ? 1.0 : 0.0);
      double dy = 2.0 * s * (v.y[k] - r) - (s == 0.0 ? 1.0 : 0.0);
      double sv = sqrt(dx * dx + dy * dy), inv = 1.0 / sv;   // one reciprocal instead of two divisions (<= 1 ulp apart)
      S[SPARSE ? 0 : k] = sv; Dx[SPARSE ? 0 : k] = dx * inv; Dy[SPARSE ? 0 : k] = dy * inv;
    }
  }
  LFPSQP_DEV void y_retract_elem(int k, double &xn, double &yn, double xb, double yb) const {  // retractions.jl:451-500
    if (idx(k) >= NA) return;
    const int kind = bkind(k);
    if (kind == 0) { xn = yn; }
    else if (kind == 1) {
      double s = bs(k), r = br(k);
      double g1 = -s, g2 = -2.0 * (yb - r), ng = sqrt(g1 * g1 + g2 * g2);
      double ux = xb - xn + g1 / ng, uy = yb - yn + g2 / ng;
      double y0 = yn - r;
      double a = s * uy * uy, b = ux + 2.0 * s * y0 * uy, c = xn + s * y0 * y0 - r;
      double a1 = -b / (2.0 * a), a2 = sqrt(b * b - 4.0 * a * c) / (2.0 * a);
      double gam = fmin(a1 + a2, a1 - a2);
      xn += gam * ux; yn += gam * uy;
    } else {
      double c = br(k), rho = sqrt(bt(k));
      double ex = xn - c, ey = yn - c, dist = sqrt(ex * ex + ey * ey);
      yn = c + rho * ey / dist;
      xn = c + rho * ex / dist;
    }
  }
  LFPSQP_DEV void y_retract(Vec &vn, int sv_base) const {  // base point (x, y) read from the stash
    LF_UNROLL for (int k = 0; k < NPL; k++) y_retract_elem(k, vn.x[k], vn.y[k], sx(sv_base, k), sy(sv_base, k));
  }
  // dest = a * fulljac' [wh ; wc] + b * dest (inequality_helper.jl:215-251)
  LFPSQP_DEV void fullJ_mulT(Vec &dest, const double *wh, const double *wc, double a, double b) const {
    LF_UNROLL for (int k = 0; k < NPL; k++) {
      double t = coldot(wc, k);
      if (INEQ) {
        double sw = gS(k) * wh[k];
        dest.x[k] = a * (t + gDx(k) * sw) + (b == 0.0 ? 0.0 : b * dest.x[k]);
        dest.y[k] = (b == 0.0 ? 0.0 : b * dest.y[k]) + a * gDy(k) * sw;
      } else dest.x[k] = a * t + (b == 0.0 ? 0.0 : b * dest.x[k]);
    }
  }

  // ---------------------------------------------------------------- Gram + Cholesky (replaces ksvd!, optimize.jl:288-302)
  LFPSQP_DEV bool factor() {
    st_fact++;
    rank = ME; pinv = false;
    double maxdiag = 0.0, Gs[MEA][MEA];
    if (ME == 1) {
      double s = 0.0;
      LF_UNROLL for (int k = 0; k < NPL; k++) { double w = INEQ ? gDy(k) * gDy(k) : 1.0; s += J[0][k] * w * J[0][k]; }
      s = sum(s);
      Lc[0][0] = s; Gs[0][0] = s; maxdiag = fmax(maxdiag, s);
    } else if (ME == 2) {
      double s00 = 0.0, s10 = 0.0, s11 = 0.0;
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        double w = INEQ ? gDy(k) * gDy(k) : 1.0;
        s00 += J[0][k] * w * J[0][k]; s10 += J[MEA - 1][k] * w * J[0][k]; s11 += J[MEA - 1][k] * w * J[MEA - 1][k];
      }
      sum3(s00, s10, s11);
      Lc[0][0] = s00; Gs[0][0] = s00; Lc[MEA - 1][0] = s10; Gs[MEA - 1][0] = s10; Gs[0][MEA - 1] = s10;
      Lc[MEA - 1][MEA - 1] = s11; Gs[MEA - 1][MEA - 1] = s11;
      maxdiag = fmax(fmax(maxdiag, s00), s11);
    }
    const double thresh = fmax(prm.eps_rank * prm.eps_rank, 1e-14 * maxdiag);
    bool ok = true;
    LF_UNROLL for (int k = 0; k < ME; k++) {
      LF_UNROLL for (int i = k; i < ME; i++) {
        double s = Lc[i][k];
        LF_UNROLL for (int t = 0; t < k; t++) s -= Lc[i][t] * Lc[k][t];
        Lc[i][k] = s;
      }
      double piv = Lc[k][k];
      if (!(piv > thresh)) { ok = false; piv = 1.0; }
      double rinv = 1.0 / sqrt(piv);
      Lc[k][k] = sqrt(piv);
      LF_UNROLL for (int i = k + 1; i < ME; i++) Lc[i][k] *= rinv;
    }
    if (ok) return true;
    // rank-deficient (optimize.jl:297-302): truncated pseudo-inverse of G through its eigen-decomposition (ME <= 2:
    // one Jacobi rotation is exact); same thresholds as batched_warp.cuh::factor_rank_deficient
    double V[MEA][MEA], ev[MEA];
    LF_UNROLL for (int a = 0; a < ME; a++) LF_UNROLL for (int b = 0; b < ME; b++) V[a][b] = (a == b) ? 1.0 : 0.0;
    if (ME == 2 && Gs[0][MEA - 1] != 0.0) {
      const double apq = Gs[0][MEA - 1], app = Gs[0][0], aqq = Gs[MEA - 1][MEA - 1];
      const double theta = (aqq - app) / (2.0 * apq);
      const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
      const double c = 1.0 / sqrt(t * t + 1.0), sn = t * c;
      V[0][0] = c; V[0][MEA - 1] = sn; V[MEA - 1][0] = -sn; V[MEA - 1][MEA - 1] = c;
      Gs[0][0] = app - t * apq; Gs[MEA - 1][MEA - 1] = aqq + t * apq;
    }
    double lmax = 0.0;
    LF_UNROLL for (int k = 0; k < ME; k++) lmax = fmax(lmax, Gs[k][k]);
    const double thr = fmax(prm.eps_rank * prm.eps_rank, 1e-13 * lmax);
    int r = 0;
    LF_UNROLL for (int k = 0; k < ME; k++) { bool keep = Gs[k][k] >= thr; ev[k] = keep ? 1.0 / Gs[k][k] : 0.0; r += keep ? 1 : 0; }
    LF_UNROLL for (int a = 0; a < ME; a++) LF_UNROLL for (int b = 0; b < ME; b++) {
      double s = 0.0;
      LF_UNROLL for (int k = 0; k < ME; k++) s += V[a][k] * ev[k] * V[b][k];
      Lc[a][b] = s;
    }
    rank = r; pinv = true;
    return true;
  }

  // v <- v - Q Q' v (optimize.jl:306-307 / :316-317, projcg.jl:59-60,:96-97); multipliers as by-product (:331-343)
  LFPSQP_DEV void project(Vec &v, bool want_mult) {
    double u[MEA];
    if (INEQ) {
      double aa[NPL], bb[NPL];
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        aa[k] = gDx(k) * v.x[k] + gDy(k) * v.y[k];
        bb[k] = gDy(k) * (gDy(k) * v.x[k] - gDx(k) * v.y[k]);
      }
      if (ME > 0) { rowdots(u, bb); solveG(u); }
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        double wj = (ME > 0) ? coldot(u, k) : 0.0;
        v.x[k] -= gDx(k) * aa[k] + gDy(k) * gDy(k) * wj;
        v.y[k] -= gDy(k) * aa[k] - gDx(k) * gDy(k) * wj;
        if (want_mult) { const double sinv = 1.0 / gS(k); lamy[k] = (-1.0 * gDx(k) * sinv) * wj + aa[k] * sinv; }
      }
    } else if (ME > 0) {
      rowdots(u, v.x); solveG(u);
      LF_UNROLL for (int k = 0; k < NPL; k++) v.x[k] -= coldot(u, k);
    }
    if (want_mult) { LF_UNROLL for (int a = 0; a < ME; a++) lam[a] = u[a]; }
  }

  // ---------------------------------------------------------------- projcg! (projcg.jl:40-121), c = 0 ; b is read from the stash
  LFPSQP_DEV void projcg(Vec &xs, int sv_b, double tol, int64_t maxit) {
    Vec r, dc, Ad, rp;
    LF_UNROLL for (int k = 0; k < NPL; k++) { xs.x[k] = 0.0; r.x[k] = -sx(sv_b, k); if (INEQ) { xs.y[k] = 0.0; r.y[k] = -sy(sv_b, k); } }
    project(r, false);
    LF_UNROLL for (int k = 0; k < NPL; k++) { dc.x[k] = -1.0 * r.x[k]; if (INEQ) dc.y[k] = -1.0 * r.y[k]; }
    int i = 0;
    const int N = INEQ ? 2 * NA : NA;
    int64_t lim = (int64_t)N + (INEQ ? NA + rank : rank); if (maxit < lim) lim = maxit;   // c has length rank / n+rank
    double rg = dot(r, r);                                                      // r == g after every projection
    while (i < lim) {
      i++;
      hess_aux(Ad, dc);
      double dAd = dot(dc, Ad);
      if (dAd <= 0.0) {                                                         // :77-82
        double nrm = sqrt(dot(dc, dc));
        LF_UNROLL for (int k = 0; k < NPL; k++) { xs.x[k] = dc.x[k] / nrm; if (INEQ) xs.y[k] = dc.y[k] / nrm; }
        st_negcurv++;
        break;
      }
      if (rg <= 0.0) break;                                                     // :87-89
      double alpha = rg / dAd;
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        xs.x[k] += alpha * dc.x[k];
        rp.x[k] = r.x[k] + alpha * Ad.x[k];
        if (INEQ) { xs.y[k] += alpha * dc.y[k]; rp.y[k] = r.y[k] + alpha * Ad.y[k]; }
      }
      r = rp;                                                                   // r becomes gp (:100-101) below
      project(r, false);                                                        // :95-97
      double rpgp = 0.0, gg = 0.0;                                              // rp.gp and gp.gp in one interleaved pass
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        rpgp += rp.x[k] * r.x[k]; gg += r.x[k] * r.x[k];
        if (INEQ) { rpgp += rp.y[k] * r.y[k]; gg += r.y[k] * r.y[k]; }
      }
      sum2(rpgp, gg);
      double beta = rpgp / rg;
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        dc.x[k] = beta * dc.x[k] - r.x[k];
        if (INEQ) dc.y[k] = beta * dc.y[k] - r.y[k];
      }
      rg = gg;                                                                  // next iteration's r.g (:84) == |g|^2
      if (sqrt(gg) < tol) break;                                                // :103-111
    }
    st_projcg += i;
  }

  // ---------------------------------------------------------------- retract!(::ProjPenalty) (retractions.jl:265-441) with pcg! (:179-246)
  // xtilde is in the stash (SV_XTIL); xnew is returned in registers
  LFPSQP_DEV int retract_pp(Vec &xnew, int *it1, int *it2) {
    int flag = 0;
    get(SV_XTIL, xnew);
    double mu = prm.mu0;
    int i = 0, pcg_total = 0;
    while (i < prm.maxiter_retract) {
      // jac!(J, cval, xnew) (:340) ; with bounds inequality_gradient! (:344), h (:350) ; curtol ; g = xnew - xtilde, g.g, h.h
      jac_fill(xnew);
      double cpart[MEA];
      c_partial(cpart, xnew);
      double hm = 0.0, gg = 0.0, hh = 0.0;
      Vec gv;
      if (INEQ) {
        inequality_gradient(xnew);
        calculate_h(cvh, xnew);
        LF_UNROLL for (int k = 0; k < NPL; k++) hm = pmax_nn(fabs(cvh[k]), hm);
      }
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        gv.x[k] = xnew.x[k] - sx(SV_XTIL, k); gg += gv.x[k] * gv.x[k];
        if (INEQ) { gv.y[k] = xnew.y[k] - sy(SV_XTIL, k); gg += gv.y[k] * gv.y[k]; hh += cvh[k] * cvh[k]; }
      }
      // one interleaved butterfly for everything this step reduces: c partial sums, max |h|, h.h, g.g
      if (ME == 1 && INEQ) {
        LF_UNROLL for (int o = LW / 2; o > 0; o >>= 1) {
          double t0 = __shfl_xor_sync(gmask, cpart[0], o), t1 = __shfl_xor_sync(gmask, hm, o), t2 = __shfl_xor_sync(gmask, hh, o),
                 t3 = __shfl_xor_sync(gmask, gg, o);
          cpart[0] += t0; hm = pmax_nn(hm, t1); hh += t2; gg += t3;
        }
      } else {
        if (ME == 2) sum2(cpart[0], cpart[MEA - 1]); else { LF_UNROLL for (int a = 0; a < ME; a++) cpart[a] = sum(cpart[a]); }
        if (INEQ) { hm = maxr(hm); sum2(hh, gg); } else gg = sum(gg);
      }
      LF_UNROLL for (int a = 0; a < ME; a++) cval[a] = cpart[a] - Fam::off(fc, a);
      double curtol = 0.0;
      LF_UNROLL for (int a = 0; a < ME; a++) curtol = pmax_nn(fabs(cval[a]), curtol);
      if (INEQ) {
        LF_UNROLL for (int a = 0; a < ME; a++) hm = pmax_nn(fabs(cvc[a]), hm);   // :352 incl. the stale tail of cvalaug
        curtol = pmax_nn(curtol, hm);
      }
      LF_UNROLL for (int a = 0; a < ME; a++) cvc[a] = cval[a];          // :356
      if (curtol < prm.eps_c) break;                                    // :359-361
      double cc = 0.0;
      LF_UNROLL for (int a = 0; a < ME; a++) cc += cvc[a] * cvc[a];
      const double prev_obj = (hh + cc) + mu * gg;                      // :366
      fullJ_mulT(gv, cvh, cvc, 1.0, mu);                                // :369
      put(SV_GV, gv); put(SV_XNEW, xnew);                               // cold during pcg!
      // pcg! (:179-246), M! = copy.  rho_k = r.r is reduced once per iteration (it is both norm(r)^2 of :235 and
      // dot(z,r) of :213) together with J r, from which J p follows by the p-recurrence (J p = J r + beta J p_old).
      Vec dx;
      int pi = 0;
      {
        Vec r, pv;
        r = gv; zero(pv);
        LF_UNROLL for (int k = 0; k < NPL; k++) { dx.x[k] = 0.0; if (INEQ) dx.y[k] = 0.0; }
        bool go = true;                                              // norm_res = Inf before the first iteration (:205)
        double rho_prev = 1.0, rho, Jr[MEA], Jp[MEA];
        {
          double a0 = 0.0, b0 = 0.0, b1 = 0.0;
          LF_UNROLL for (int k = 0; k < NPL; k++) {
            a0 += r.x[k] * r.x[k]; if (INEQ) a0 += r.y[k] * r.y[k];
            if (ME > 0) b0 += J[0][k] * r.x[k];
            if (ME > 1) b1 += J[MEA - 1][k] * r.x[k];
          }
          if (ME == 2) { sum3(a0, b0, b1); Jr[0] = b0; Jr[MEA - 1] = b1; } else if (ME == 1) { sum2(a0, b0); Jr[0] = b0; } else a0 = sum(a0);
          rho = a0;
          LF_UNROLL for (int a = 0; a < MEA; a++) Jp[a] = 0.0;
        }
        while (go && pi < prm.maxiter_pcg) {                        // norm_res > tol (:207)
          const double beta = rho / rho_prev;
          LF_UNROLL for (int k = 0; k < NPL; k++) { pv.x[k] = r.x[k] + beta * pv.x[k]; if (INEQ) pv.y[k] = r.y[k] + beta * pv.y[k]; }
          LF_UNROLL for (int a = 0; a < ME; a++) Jp[a] = Jr[a] + beta * Jp[a];
          Vec z;
          double pz = 0.0;
          LF_UNROLL for (int k = 0; k < NPL; k++) {                  // z = fulljac'(fulljac p) + mu p ; p.z
            const double t = coldot(Jp, k);
            if (INEQ) {
              const double th = gS(k) * (gDx(k) * pv.x[k] + gDy(k) * pv.y[k]);
              const double sw = gS(k) * th;
              z.x[k] = 1.0 * (t + gDx(k) * sw) + mu * pv.x[k];
              z.y[k] = mu * pv.y[k] + 1.0 * gDy(k) * sw;
            } else z.x[k] = 1.0 * t + mu * pv.x[k];
          }
          LF_UNROLL for (int k = 0; k < NPL; k++) pz += pv.x[k] * z.x[k];
          if (INEQ) { LF_UNROLL for (int k = 0; k < NPL; k++) pz += pv.y[k] * z.y[k]; }
          const double alpha = rho / sum(pz);
          double a0 = 0.0, b0 = 0.0, b1 = 0.0;
          LF_UNROLL for (int k = 0; k < NPL; k++) {
            dx.x[k] += alpha * pv.x[k]; r.x[k] -= alpha * z.x[k]; a0 += r.x[k] * r.x[k];
            if (ME > 0) b0 += J[0][k] * r.x[k];
            if (ME > 1) b1 += J[MEA - 1][k] * r.x[k];
            if (INEQ) { dx.y[k] += alpha * pv.y[k]; r.y[k] -= alpha * z.y[k]; a0 += r.y[k] * r.y[k]; }
          }
          if (ME == 2) { sum3(a0, b0, b1); Jr[0] = b0; Jr[MEA - 1] = b1; } else if (ME == 1) { sum2(a0, b0); Jr[0] = b0; } else a0 = sum(a0);
          rho_prev = rho; rho = a0;
          go = rho > pcg_rho_stop;                                   // == sqrt(rho) > eps_c (:235)
          pi++;
        }
      }
      pcg_total += pi;
      if (pi == prm.maxiter_pcg) { get(SV_XNEW, xnew); flag = 2; break; }   // :240-243, :377-381
      // inner Armijo (:384-426): p = xnew (stays in the stash) ; xnew -= dx ; g = xnew - xtilde
      double ard = 0.0, s2 = 0.0;
      LF_UNROLL for (int k = 0; k < NPL; k++) ard += sx(SV_GV, k) * dx.x[k];
      if (INEQ) { LF_UNROLL for (int k = 0; k < NPL; k++) ard += sy(SV_GV, k) * dx.y[k]; }
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        xnew.x[k] = sx(SV_XNEW, k) - 1.0 * dx.x[k]; { const double t = xnew.x[k] - sx(SV_XTIL, k); s2 += t * t; }
        if (INEQ) { xnew.y[k] = sy(SV_XNEW, k) - 1.0 * dx.y[k]; const double t = xnew.y[k] - sy(SV_XTIL, k); s2 += t * t; }
      }
      double alpha = 1.0;
      c_partial(cpart, xnew);                                           // :392
      double h2 = 0.0;
      if (INEQ) { calculate_h(cvh, xnew); LF_UNROLL for (int k = 0; k < NPL; k++) h2 += cvh[k] * cvh[k]; }
      if (ME == 1 && INEQ) {
        LF_UNROLL for (int o = LW / 2; o > 0; o >>= 1) {
          double t0 = __shfl_xor_sync(gmask, cpart[0], o), t1 = __shfl_xor_sync(gmask, ard, o), t2 = __shfl_xor_sync(gmask, s2, o),
                 t3 = __shfl_xor_sync(gmask, h2, o);
          cpart[0] += t0; ard += t1; s2 += t2; h2 += t3;
        }
      } else {
        if (ME == 2) sum2(cpart[0], cpart[MEA - 1]); else { LF_UNROLL for (int a = 0; a < ME; a++) cpart[a] = sum(cpart[a]); }
        if (INEQ) sum3(ard, s2, h2); else sum2(ard, s2);
      }
      const double ar_dot = -ard;
      double dist2 = s2;
      LF_UNROLL for (int a = 0; a < ME; a++) { cval[a] = cpart[a] - Fam::off(fc, a); cvc[a] = cval[a]; }
      int armijo_count = 0;
      while (true) {
        double c2 = 0.0;
        LF_UNROLL for (int a = 0; a < ME; a++) c2 += cvc[a] * cvc[a];
        if (!((h2 + c2) + mu * dist2 > prev_obj + 1e-4 * alpha * ar_dot)) break;   // :403
        alpha /= 2; s2 = 0.0;
        LF_UNROLL for (int k = 0; k < NPL; k++) {
          xnew.x[k] = sx(SV_XNEW, k) - alpha * dx.x[k]; { const double t = xnew.x[k] - sx(SV_XTIL, k); s2 += t * t; }
          if (INEQ) { xnew.y[k] = sy(SV_XNEW, k) - alpha * dx.y[k]; const double t = xnew.y[k] - sy(SV_XTIL, k); s2 += t * t; }
        }
        h2 = 0.0;
        if (INEQ) { calculate_h(cvh, xnew); LF_UNROLL for (int k = 0; k < NPL; k++) h2 += cvh[k] * cvh[k]; sum2(s2, h2); }   // :410-417: only the bound part is refreshed, the c-part stays frozen
        else s2 = sum(s2);
        dist2 = s2;
        armijo_count++; st_bt++;
        if (armijo_count == 100) { flag = 3; break; }
      }
      i++;
      double nn = h2;
      LF_UNROLL for (int a = 0; a < ME; a++) nn += cvc[a] * cvc[a];
      mu = fmin(mu * 0.1, sqrt(nn));                                    // :431
    }
    if (i == prm.maxiter_retract) flag = 1;
    *it1 = i; *it2 = pcg_total;
    return flag;
  }

  // ---------------------------------------------------------------- retract!(::NR) (retractions.jl:75-177), Cholesky-QR basis
  // xtilde and the base point x are in the stash (SV_XTIL, SV_X)
  LFPSQP_DEV int retract_nr(Vec &xnew, int *it1) {
    double D[MEA][MEA], t1[MEA], t2[MEA], dcv[MEA];
    get(SV_XTIL, xnew);
    if (INEQ) y_retract(xnew, SV_X);
    c_aux(cval, xnew);
    LF_UNROLL for (int c = 0; c < ME; c++)        // D0 = L^-1
      LF_UNROLL for (int i = 0; i < ME; i++) {
        double s = (i == c) ? 1.0 : 0.0;
        LF_UNROLL for (int t = 0; t < i; t++) if (t >= c) s -= Lc[i][t] * D[t][c];
        D[i][c] = (i < c) ? 0.0 : s / Lc[i][i];
      }
    int i = 0;
    while (i < prm.maxiter_retract) {
      double cm = 0.0;
      LF_UNROLL for (int a = 0; a < ME; a++) cm = pmax_nn(fabs(cval[a]), cm);
      if (cm < prm.eps_c) break;
      LF_UNROLL for (int a = 0; a < ME; a++) { double s = 0.0; LF_UNROLL for (int b = 0; b < ME; b++) s += D[a][b] * cval[b]; t1[a] = -s; }
      double yv[MEA];                              // xnew += Q delta, Q = PJct L^-T
      LF_UNROLL for (int a = 0; a < ME; a++) yv[a] = t1[a];
      LF_UNROLL for (int k = ME - 1; k >= 0; k--) { double s = yv[k]; LF_UNROLL for (int t = k + 1; t < ME; t++) s -= Lc[t][k] * yv[t]; yv[k] = s / Lc[k][k]; }
      LF_UNROLL for (int k = 0; k < NPL; k++) {
        double wj = coldot(yv, k);
        if (INEQ) { xnew.x[k] += gDy(k) * gDy(k) * wj; xnew.y[k] -= gDx(k) * gDy(k) * wj; } else xnew.x[k] += wj;
      }
      if (INEQ) y_retract(xnew, SV_X);
      c_aux(t2, xnew);
      LF_UNROLL for (int a = 0; a < ME; a++) { dcv[a] = t2[a] - cval[a]; cval[a] = t2[a]; }
      LF_UNROLL for (int a = 0; a < ME; a++) { double s = 0.0; LF_UNROLL for (int b = 0; b < ME; b++) s += D[b][a] * t1[b]; t2[a] = s; }
      double den = 0.0;
      LF_UNROLL for (int a = 0; a < ME; a++) den += t2[a] * dcv[a];
      LF_UNROLL for (int a = 0; a < ME; a++) { double s = 0.0; LF_UNROLL for (int b = 0; b < ME; b++) s += D[a][b] * dcv[b]; t1[a] -= s; }
      double al = 1.0 / den;
      LF_UNROLL for (int a = 0; a < ME; a++) LF_UNROLL for (int b = 0; b < ME; b++) D[a][b] += al * t1[a] * t2[b];
      i++;
    }
    *it1 = i;
    return (i == prm.maxiter_retract) ? 1 : 0;
  }

  // ---------------------------------------------------------------- the driver (optimize.jl:176-443)
  LFPSQP_DEV void run(const BatchedArgs &A, int64_t k) {
    fc.prm = A.fam_params ? A.fam_params + k * A.fam_stride : nullptr;
    st_projcg = st_negcurv = st_trials = st_rout = st_rpcg = st_bt = st_newton = st_fact = st_feval = 0; status = 0;
    rank = ME; pinv = false;
    LF_UNROLL for (int s = 0; s < NPL; s++) {
      int j = idx(s);
      LF_UNROLL for (int q = 0; q < KP; q++) ep[s][q] = 0.0;
      if (j < n) Fam::load(fc, j, ep[s]);
      x.x[s] = (j < n) ? A.x0[k * n + j] : 0.0;
      if (INEQ) x.y[s] = 0.0;
      cvh[s] = 0.0; lamy[s] = 0.0;
    }
    if (INEQ) init_line_gradients();
    LF_UNROLL for (int a = 0; a < MEA; a++) { cvc[a] = 0.0; cval[a] = 0.0; lam[a] = 0.0; }
    if (ME > 0 && p > 0) {  // slack start values s0 = d(x0) (optimize.jl:26-28): c_aux with s = 0 gives d(x0) in rows >= m
      double cv0[MEA];
      c_aux(cv0, x);
      LF_UNROLL for (int s = 0; s < NPL; s++) { int j = idx(s); LF_UNROLL for (int a = 0; a < ME; a++) if (a >= m && j == n + (a - m)) x.x[s] = cv0[a]; }
    }
    if (INEQ) generate_initial_y(x);
    int64_t it = 0, nobj = 0;
    double f_diff = INFINITY, step_diff = INFINITY, kkt_diff = INFINITY, prev_grad_norm = 0.0;
    double fval = f_aux(x);
    if (lane == 0 && nobj < A.H) A.obj_hist[k * A.H + nobj] = fval;
    nobj++;
    if (ME > 0) c_aux(cval, x);
    int cond = LFPSQP_F_TOL, last_flag = 0;
    while (true) {
      {
        Vec d;   // d = -grad f (optimize.jl:259-262); the gradient itself is re-evaluated for ar_dot instead of being kept
        LF_UNROLL for (int s = 0; s < NPL; s++) {
          double e[KP] = {0.0};
          if (user(s)) eload(s, e);
          const double gs = user(s) ? Fam::g(fc, idx(s), x.x[s], e) : 0.0;
          d.x[s] = -1.0 * gs;
          if (INEQ) d.y[s] = -0.0;
        }
        if (A.noise) {                                                           // :264-273, caller-supplied noise rows
          const double nc = noise_coef(prm, it, A.noise_T);
          if (nc != 0.0) {
            const int Nw = INEQ ? 2 * NA : NA;
            const double *nz = A.noise + ((int64_t)k * A.noise_T + it) * Nw;
            LF_UNROLL for (int s = 0; s < NPL; s++) {
              if (idx(s) < NA) { d.x[s] += nc * nz[idx(s)]; if (INEQ) d.y[s] += nc * nz[NA + idx(s)]; }
            }
          }
        }
        if (INEQ) inequality_gradient(x);
        if (ME > 0) {
          jac_aux(cval, x);
          factor();
          if (pinv) status |= LFPSQP_ST_RANK_DEFICIENT;   // informational: truncated path of optimize.jl:297-302
        }
        project(d, true);
        double km = 0.0;
        LF_UNROLL for (int s = 0; s < NPL; s++) { km = pmax_nn(fabs(d.x[s]), km); if (INEQ) km = pmax_nn(fabs(d.y[s]), km); }
        kkt_diff = maxr(km);                                                     // :320
        if (f_diff <= prm.eps_f) { cond = LFPSQP_F_TOL; break; }
        else if (step_diff <= prm.eps_x) { cond = LFPSQP_X_TOL; break; }
        else if (it >= prm.maxiter) { cond = LFPSQP_MAX_ITER; break; }
        else if (kkt_diff <= prm.eps_kkt) { cond = LFPSQP_KKT_TOL; break; }
        if (!(kkt_diff == kkt_diff)) { status |= LFPSQP_ST_NONFINITE; cond = LFPSQP_MAX_ITER; break; }
        put(SV_D, d);
        if (prm.do_newton) {
          double gn = sqrt(dot(d, d));
          double tol = prm.tn_kappa * fmin(1.0, gn / prev_grad_norm) * gn;
          prev_grad_norm = gn;
          Vec nd;
          projcg(nd, SV_D, tol, prm.tn_maxiter);
          double s = 0.0;
          LF_UNROLL for (int q = 0; q < NPL; q++) s += nd.x[q] * sx(SV_D, q);
          if (INEQ) { LF_UNROLL for (int q = 0; q < NPL; q++) s += nd.y[q] * sy(SV_D, q); }
          if (sum(s) > 0.0) { put(SV_D, nd); st_newton++; }
        }
      }
      int kind;
      if (ME > 0) kind = (rank == ME && !prm.do_project_retract) ? 2 : 3; else kind = INEQ ? 1 : 0;
      // armijo! (linesearch.jl:32-89) ; x and d stay in the stash while the retraction runs
      double alpha = prm.alpha, newf = 0.0;
      f_diff = INFINITY; step_diff = INFINITY;
      double ar_dot = 0.0;                                                       // d.g (the y-half of g is zero)
      LF_UNROLL for (int s = 0; s < NPL; s++) {
        double e[KP] = {0.0};
        if (user(s)) eload(s, e);
        const double gs = user(s) ? Fam::g(fc, idx(s), x.x[s], e) : 0.0;
        ar_dot += sx(SV_D, s) * gs;
      }
      ar_dot = sum(ar_dot);
      put(SV_X, x);
      int flag = 0;
      Vec xnew;
      while (step_diff > prm.eps_x) {
        LF_UNROLL for (int s = 0; s < NPL; s++) { sx(SV_XTIL, s) = sx(SV_X, s) + alpha * sx(SV_D, s); if (INEQ) sy(SV_XTIL, s) = sy(SV_X, s) + alpha * sy(SV_D, s); }
        int i1 = 0, i2 = 0;
        if (kind == 0) { get(SV_XTIL, xnew); flag = 0; }
        else if (kind == 1) { get(SV_XTIL, xnew); y_retract(xnew, SV_X); flag = 0; }
        else if (kind == 2) flag = retract_nr(xnew, &i1);
        else flag = retract_pp(xnew, &i1, &i2);
        st_rout += i1; st_rpcg += i2; st_trials++;
        // linesearch.jl:57-60 has no lower bound on alpha in this branch: when the retraction fails at EVERY alpha the
        // reference spins forever once alpha has underflowed to 0.  Stop at the floor the other branch uses (:82-85):
        // flag 98, LFPSQP_ST_NONFINITE.
        if (flag > 0) { if (alpha < 1e-100) { flag = 98; break; } alpha *= prm.s; continue; }
        newf = f_aux(xnew);
        double s2 = 0.0;
        LF_UNROLL for (int s = 0; s < NPL; s++) { double t = xnew.x[s] - sx(SV_X, s); s2 += t * t; }   // first n_A entries (:66)
        step_diff = sqrt(sum(s2));
        f_diff = fabs(newf - fval);
        if (prm.disable_linesearch) break;
        if ((newf - fval) <= prm.sigma * alpha * ar_dot) break;
        alpha *= prm.s;
        if (alpha < 1e-100) { flag = 99; break; }
      }
      last_flag = flag;
      if (flag == 98) { get(SV_X, x); status |= LFPSQP_ST_NONFINITE; cond = LFPSQP_MAX_ITER; break; }
      x = xnew;
      fval = newf;
      if (lane == 0 && nobj < A.H) A.obj_hist[k * A.H + nobj] = fval;
      nobj++;
      it++;
    }
    LF_UNROLL for (int s = 0; s < NPL; s++) { int j = idx(s); if (j < n) A.x_out[k * n + j] = x.x[s]; }
    if (lane == 0) {
      LF_UNROLL for (int a = 0; a < ME; a++) A.lambda[k * ME + a] = lam[a];
      A.obj_len[k] = nobj;
      lfpsqp_term t; t.condition = cond; t.status = status; t.f_diff = f_diff; t.step_diff = step_diff;
      t.kkt_diff = kkt_diff; t.iter = it;
      A.term[k] = t;
      if (A.stats) {
        lfpsqp_stats st;
        st.projcg_iters = st_projcg; st.projcg_negcurv = st_negcurv; st.armijo_trials = st_trials; st.retract_outer = st_rout;
        st.retract_pcg = st_rpcg; st.pp_backtracks = st_bt; st.newton_accepted = st_newton; st.factorizations = st_fact;
        st.f_evals = st_feval; st.flag_last = last_flag;
        A.stats[k] = st;
      }
    }
  }
};

// Persistent CTAs of REG_NT threads = REG_NT / LW lane groups; every group pulls instance indices from a global counter
// until the batch is drained (absorbs the per-instance iteration-count variance).  The groups of a warp leave the loop
// together.  MINB = resident CTAs per SM the register allocation is capped for (3 -> 168 registers, 2 -> 255).
// SPARSE, HEAD: see RegSolver.
constexpr int REG_NT = 128;
template <class Fam, int LW, int NPL, int ME, bool INEQ, bool SPARSE, int HEAD, int MINB>
__global__ void __launch_bounds__(REG_NT, MINB) batched_reg_kernel(const BatchedArgs A) {
  using RS = RegSolver<Fam, LW, NPL, ME, INEQ, SPARSE, HEAD>;
  extern __shared__ double smem[];
  const int lane32 = threadIdx.x & 31;
  int sub = lane32 % LW;
  unsigned gmask = (LW == 32) ? 0xffffffffu : (((1u << (LW & 31)) - 1u) << (lane32 / LW * LW));
  const int NA = A.n + A.p;
  double *bnd = smem;
  constexpr int NB = INEQ ? 5 * RS::NAP : 0;
  for (int i = threadIdx.x; i < NB; i += blockDim.x) {
    const int a = i / RS::NAP, j = i % RS::NAP;
    bnd[i] = (j < NA) ? A.bnd[a * NA + j] : 0.0;
  }
  __syncthreads();
  double *stash = smem + NB + (size_t)(threadIdx.x / 32) * RS::GPW * RS::STASH_DOUBLES + lane32;
  RS S(sub, gmask, A.prm, A.n, A.m, A.p, bnd, stash);
  for (;;) {
    unsigned long long k = 0;
    if (sub == 0) k = atomicAdd(A.work_counter, 1ULL);
    k = __shfl_sync(gmask, k, 0, LW);
    const bool active = (int64_t)k < A.B;
    if (!__any_sync(0xffffffffu, active)) break;
    if (active) S.run(A, (int64_t)k);
  }
}

}  // namespace lfpsqp
