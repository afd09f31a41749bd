/*
 * lfpsqp_b200.h -- C ABI of the B200-native LFPSQP hot path (liblfpsqp_b200.so).
 *
 * This is the drop-in boundary: the symbols a Julia maintainer binds with `ccall` in place of the pure-Julia
 * hot path of LFPSQP.jl (the existing FFI style is src/la_helper.jl:22-28, :37-43: plain C symbols, arrays as
 * Ptr{Float64}, status by integer).  Every array is dense, Float64, host memory unless the name ends in `_dev`.
 * Matrices follow Julia's column-major convention at the boundary: an (n x B) batch is instance-major in memory
 * (instance k occupies [k*n, (k+1)*n)).  The constraint Jacobian is held on the device as J (m x n) ROW-major,
 * which is byte-identical to the reference's `Jct` (n x m column-major, src/optimize.jl:190).
 *
 * Julia closures cannot run on the device, so f / c! / d! and their derivatives are REGISTERED DEVICE FAMILIES
 * (family id + parameter blob) -- the contract they implement is the one src/autodiff_generators.jl produces:
 * grad!(g,x) (:7-9), jac!(Jc,cval,x) which also writes cval (:40-42), hess_lag_vec!(dest,src,x,lambda) (:80-104).
 *
 * Return codes: 0 ok; <0 argument errors mirroring the reference's error() calls; CUDA errors are mapped to
 * LFPSQP_ERR_CUDA.  Message via lfpsqp_last_error().  Algorithmic failures are in-band per-instance flags.
 * Calls block until results are in the caller's buffers.  One ctx per host thread (a ctx is not re-entrant).
 */
#ifndef LFPSQP_B200_H
#define LFPSQP_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LFPSQP_OK 0
#define LFPSQP_ERR_ARG (-1)        /* bad sizes: optimize.jl:19-21, :144-148 ; inequality_helper.jl:42-44 */
#define LFPSQP_ERR_BOUNDS (-2)     /* "Infeasible: lower bounds cannot be greater than upper bounds" optimize.jl:160-162 */
#define LFPSQP_ERR_FAMILY (-3)     /* unknown family / family does not support these sizes */
#define LFPSQP_ERR_UNSUPPORTED (-4)/* beta>0 noise (optimize.jl:264-273), user callback (:432-434) */
#define LFPSQP_ERR_CUDA (-5)
#define LFPSQP_ERR_NOMEM (-6)
#define LFPSQP_ERR_COMM (-7)
#define LFPSQP_ERR_CALLBACK (-8)   /* a host callback returned non-zero (the Julia wrapper rethrows the stored exception) */

/* LFPSQPParams, src/LFPSQP.jl:57-81 (same defaults: lfpsqp_default_params). disp/callback are host-side
 * cosmetics of the reference and are ignored by the device path. */
typedef struct {
  double alpha, beta;
  int64_t t_beta;
  double s, sigma, eps_c, eps_f, eps_x, eps_kkt, eps_rank;
  int64_t maxiter, maxiter_retract, maxiter_pcg;
  double mu0;
  int32_t disable_linesearch, do_project_retract, disp, linesearch /*0 armijo, 1 exact*/, do_newton;
  int32_t _pad;
  int64_t tn_maxiter;
  double tn_kappa;
  int64_t callback_period;
} lfpsqp_params;

/* TerminationCondition, src/LFPSQP.jl:37-43 */
enum { LFPSQP_F_TOL = 0, LFPSQP_X_TOL = 1, LFPSQP_KKT_TOL = 2, LFPSQP_MAX_ITER = 3, LFPSQP_ARMIJO_ERROR = 4 };

/* per-instance status bits (in-band; 0 = the path is the reference's path) */
#define LFPSQP_ST_RANK_DEFICIENT 1 /* the projected Jacobian lost rank at some iterate: informational -- the truncated path of
                                      optimize.jl:297-302 was taken (eigen-decomposition of J W J', truncated pseudo-inverse;
                                      batched mode: in shared memory, large-n mode: one-sided Jacobi on the device) */
#define LFPSQP_ST_NONFINITE 2      /* a non-finite iterate, or the retraction failed at every step length down to alpha < 1e-100
                                      (flag_last = 98; the reference spins forever there, src/linesearch.jl:57-60) */

/* TerminationInfo, src/LFPSQP.jl:45-51 : {Int32 enum, 3 x Float64, Int64}; the enum's padding carries status */
typedef struct {
  int32_t condition;
  int32_t status;
  double f_diff, step_diff, kkt_diff;
  int64_t iter;
} lfpsqp_term;

/* optional per-instance counters (NULL to skip). flag_last = last line-search/retraction flag (linesearch.jl:32-89) */
typedef struct {
  int64_t projcg_iters, projcg_negcurv, armijo_trials, retract_outer, retract_pcg, pp_backtracks;
  int64_t newton_accepted, factorizations, f_evals;
  int64_t flag_last;
} lfpsqp_stats;

/* registered device families (the benchmark problem families of BASELINE.json + the reference's test systems) */
enum {
  LFPSQP_FAM_ROSENBROCK = 0, /* README.md:18-22; n=2, m=p=0; no params */
  LFPSQP_FAM_README_EQ = 1,  /* README.md:41-54; f=x.x, c=x[1]-0.75; m=1 */
  LFPSQP_FAM_README_INEQ = 2,/* README.md:57-76; f=coeff.x, d=x.x-1; p=1; params = coeff[n] per instance */
  LFPSQP_FAM_THOMSON = 3,    /* n=3N, f=sum_{i<j} 1/|xi-xj|, c_i=|x_i|^2-1, m=N */
  LFPSQP_FAM_DIAGQUAD = 4,   /* c_i = 1/2 sum_j Q_ij x_j^2 + A_i.x - b_i ; f = 1/2 sum_j w_j (x_j-xt_j)^2
                                params = [Q (m x n row-major), A (m x n row-major), b(m), xt(n), w(n)] */
  LFPSQP_FAM_SIN = 5,        /* test/test_retractions.jl:34-54: c_i = x[2i]-sin(x[2i-1]); f=1/2|x-t|^2; params=t[n] */
  LFPSQP_FAM_BOXQUAD = 6,    /* f=|x-t|^2, optional c=a.x-b (m in {0,1}); params=[t(n), a(n), b] */
  LFPSQP_FAM_COUNT = 7,
  LFPSQP_FAM_HOST = 100      /* generic problem: f / grad! / c! / jac! / hess_lag_vec! are HOST callbacks (lfpsqp_host_callbacks);
                                large-n mode, one GPU.  The linear algebra runs on the device, the callbacks on the host. */
};

/*
 * Dense QCQP (batched mode only; lfpsqp_solve_large / lfpsqp_large_setup return LFPSQP_ERR_FAMILY for it):
 *   f(x)   = 1/2 x'P x + q.x + r
 *   c_i(x) = 1/2 x'Qc_i x + Ac_i.x - bc_i = 0      i < m
 *   d_k(x) = 1/2 x'Qd_k x + Ad_k.x - bd_k <= 0     k < p
 * Each array has a batch stride in doubles: 0 = shared by the whole batch, otherwise instance k reads ptr + k*stride
 * (stride >= the array's element count).  NULL = all zero.  Matrices are n x n, symmetric, row-major (identical to
 * column-major); stacks are m (or p) such matrices back to back.  Ac / Ad are m x n / p x n row-major (row i = a_i).
 * lfpsqp_solve_batched takes host pointers and checks that every matrix is exactly symmetric; lfpsqp_solve_batched_dev
 * takes device pointers and requires symmetric matrices.  The struct itself is host memory in both cases.
 */
typedef struct {
  const double *P;  int64_t P_stride;    /* n*n   */
  const double *q;  int64_t q_stride;    /* n     */
  const double *r;  int64_t r_stride;    /* 1     */
  const double *Qc; int64_t Qc_stride;   /* m*n*n */
  const double *Ac; int64_t Ac_stride;   /* m*n   */
  const double *bc; int64_t bc_stride;   /* m     */
  const double *Qd; int64_t Qd_stride;   /* p*n*n */
  const double *Ad; int64_t Ad_stride;   /* p*n   */
  const double *bd; int64_t bd_stride;   /* p     */
} lfpsqp_qcqp;
#define LFPSQP_FAM_QCQP 101   /* fam_params = (const double*)(const lfpsqp_qcqp*), fam_stride must be 0 */

/*
 * Host callbacks of the explicit-derivative core optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m, param)
 * (src/optimize.jl:119-143).  Conventions are the reference's (src/autodiff_generators.jl:7-9, :40-42, :80-104):
 * x is the first n entries of the working vector (optimize.jl:259 passes view(x, 1:n)); jac! fills Jc (m x n,
 * COLUMN-major: Jc[i + j*m], optimize.jl:189) AND cval; hess_lag_vec! writes dest = (Hess f + sum_i lam_i Hess c_i) src.
 * Every callback returns 0 on success; non-zero aborts the solve with LFPSQP_ERR_CALLBACK.  All pointers are host
 * memory owned by the library (pinned), valid only during the call.  c and jac may be NULL iff m == 0.
 * callback (optional) is param.callback(i, x) (optimize.jl:432-434; x has length n, or 2n with finite bounds), called when
 * i % param.callback_period == 0.  randn (optional) must fill buf with standard normals (randn!(tmp_n), optimize.jl:264-273):
 * it is what makes beta > 0 reproducible from the caller's own RNG stream; beta > 0 without it is LFPSQP_ERR_UNSUPPORTED.
 */
typedef struct {
  void *user;
  int (*f)(void *user, const double *x, int64_t n, double *fval);
  int (*grad)(void *user, double *g, const double *x, int64_t n);
  int (*c)(void *user, double *cval, const double *x, int64_t n, int64_t m);
  int (*jac)(void *user, double *Jc, double *cval, const double *x, int64_t n, int64_t m);
  int (*hess_lag_vec)(void *user, double *dest, const double *src, const double *x, const double *lam, int64_t n, int64_t m);
  int (*callback)(void *user, int64_t iter, const double *x_aug, int64_t n_aug);
  int (*randn)(void *user, double *buf, int64_t n_aug);
} lfpsqp_host_callbacks;

typedef struct lfpsqp_ctx lfpsqp_ctx;

const char *lfpsqp_version(void);
void lfpsqp_default_params(lfpsqp_params *p);                      /* src/LFPSQP.jl:57-81 */
int lfpsqp_ctx_create(int device, lfpsqp_ctx **out);               /* fails loudly (LFPSQP_ERR_CUDA) without a GPU */
void lfpsqp_ctx_destroy(lfpsqp_ctx *ctx);
/* Multi-GPU context (SURVEY.md 8b "create context (device list)"): lfpsqp_solve_batched on such a ctx shards the B instances
 * into contiguous, balanced ranges over the listed devices from ONE host call -- one host thread, one stream pipeline and one
 * device arena per GPU, no collective (the instances are independent); results land in disjoint slices of the caller's
 * arrays.  Every other entry point runs on devices[0].  Each device may be listed once.  destroy releases all of them. */
int lfpsqp_ctx_create_multi(const int *devices, int ndev, lfpsqp_ctx **out);
int lfpsqp_ctx_device_count(lfpsqp_ctx *ctx);
const char *lfpsqp_last_error(lfpsqp_ctx *ctx);                    /* ctx may be NULL: last error of ctx_create */
/* run on a caller-owned stream (e.g. torch's current stream) instead of the ctx's own; NULL restores it */
int lfpsqp_ctx_set_stream(lfpsqp_ctx *ctx, void *cuda_stream);
/* Stochastic perturbation beta > 0 (src/optimize.jl:264-273) on the device-family paths: the reference adds
 * beta * max(1 - i / t_beta, 0) * randn!(tmp_n) to d at every outer iteration i.  The caller draws that sequence from ITS OWN RNG
 * (Julia: randn(N, T) is exactly the stream T successive randn!(tmp_n) calls consume) and hands it over before the solve:
 * noise[(k * T + i) * N + j] = entry j of the draw of iteration i of instance k; N = working dimension (n + p, doubled when bounds
 * or d! are present: optimize.jl:172), B = instances of the next lfpsqp_solve_batched* call (large-n: B = 1, N = this rank's
 * working entries [x-half | y-half]).  Iterations i >= T add no noise (with t_beta > 0, T = t_beta rows cover the whole ramp).
 * The pointer must stay valid until the solve returns; NULL clears it.  Without it beta > 0 is LFPSQP_ERR_UNSUPPORTED. */
int lfpsqp_ctx_set_noise(lfpsqp_ctx *ctx, const double *noise, int64_t T, int64_t N, int64_t B);
/* device time (ms, CUDA events on the launching stream) and launch count of the kernels of the last solve call */
double lfpsqp_last_kernel_ms(lfpsqp_ctx *ctx);
int64_t lfpsqp_last_launches(lfpsqp_ctx *ctx);
/* which batched kernel the last lfpsqp_solve_batched* call launched: out4 = {kind, LW, NPL, SPARSE} with kind 0 = one thread
 * per instance (LW = 1), 1 = shared-memory warp solver (LW = 32), 2 = register-resident solver (LW lanes per instance, NPL
 * elements per lane, SPARSE = 1 for the one-exception-per-lane bound layout); kind = -1 when the last call launched none */
int lfpsqp_last_kernel(lfpsqp_ctx *ctx, int *out4);

/*
 * Batched mode: B independent instances of optimize(f, c!, d!, x0, xl, xu, m, p, param)  (src/optimize.jl:83-85 and
 * the methods it forwards to, :13-71, :88-104, :119-443), solved in lockstep on one GPU, one warp (or one thread for
 * tiny unconstrained problems) per instance.
 *   fam_params : per-instance parameter blobs, instance k at fam_params + k*fam_stride (fam_stride 0 = shared);
 *                LFPSQP_FAM_QCQP: a const lfpsqp_qcqp* cast to const double*, with fam_stride = 0
 *   x0         : n x B ; xl, xu : n (shared by the batch) or NULL (= `nothing`)
 *   x_out      : n x B ; obj_hist : H x B (first min(len,H) objective values) ; obj_len : B (iters+1)
 *   lambda     : (m+p) x B (untruncated, optimize.jl:67-70) ; term : B ; stats : B or NULL
 */
int lfpsqp_solve_batched(lfpsqp_ctx *ctx, int family, int64_t n, int64_t m, int64_t p, int64_t B,
                         const double *fam_params, int64_t fam_stride, const double *x0, const double *xl,
                         const double *xu, const lfpsqp_params *params, double *x_out, double *obj_hist, int64_t H,
                         int64_t *obj_len, double *lambda, lfpsqp_term *term, lfpsqp_stats *stats);
/* same with every array already resident in device memory (xl/xu stay host: they are n doubles of setup data) */
int lfpsqp_solve_batched_dev(lfpsqp_ctx *ctx, int family, int64_t n, int64_t m, int64_t p, int64_t B,
                             const double *fam_params_dev, int64_t fam_stride, const double *x0_dev, const double *xl,
                             const double *xu, const lfpsqp_params *params, double *x_out_dev, double *obj_hist_dev,
                             int64_t H, int64_t *obj_len_dev, double *lambda_dev, lfpsqp_term *term_dev,
                             lfpsqp_stats *stats_dev);

/*
 * Large-n mode: ONE instance with a dense m x n constraint Jacobian, host-orchestrated whole-GPU kernels
 * (FP64 DMMA Gram + blocked Cholesky replace ksvd!, src/la_helper.jl:8-34 / optimize.jl:291-293; streaming passes over
 * J replace kgemv!, la_helper.jl:36-44).  Families: LFPSQP_FAM_DIAGQUAD, LFPSQP_FAM_THOMSON,
 * LFPSQP_FAM_HOST (params = const lfpsqp_host_callbacks*); LFPSQP_FAM_QCQP is LFPSQP_ERR_FAMILY here.  Finite bounds xl <= x <= xu run the reference's 2n-variable
 * embedding (src/inequality_helper.jl): lfpsqp_large_set_bounds after lfpsqp_large_setup, or the xl/xu arguments of
 * lfpsqp_solve_large / lfpsqp_solve_host.  projcg! on diagonal Lagrangian Hessians and pcg! run as persistent cooperative
 * kernels (large_fused.cu); LFPSQP_FUSED_PROJCG=0 in the environment selects the launch-per-phase loops.
 * Column sharding: with a communicator (lfpsqp_comm_init) rank g owns columns [col0, col0+n_loc) of J and the same
 * entries of every n-vector; m-vectors and the m x m factor are replicated; only the Gram, the m-vector J v and the
 * CG scalars are all-reduced.  Without a communicator col0 = 0, n_loc = n.
 */
/* optimize(f, c!, x0, xl, xu, m, param) for one large instance on one GPU (fam_params, x0, xl, xu: host; xl/xu may be NULL) */
int lfpsqp_solve_large(lfpsqp_ctx *ctx, int family, int64_t n, int64_t m, const double *fam_params, const double *x0,
                       const double *xl, const double *xu, const lfpsqp_params *params, double *x_out, double *obj_hist,
                       int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term, lfpsqp_stats *stats);
/* two-step form: bind the (sharded) problem once, then solve / probe it.  DIAGQUAD params = this rank's shard
 * [Q_loc (m x n_loc row-major), A_loc (m x n_loc), b (m), xt_loc (n_loc), w_loc (n_loc)], host or device memory. */
int lfpsqp_large_setup(lfpsqp_ctx *ctx, int family, int64_t n_global, int64_t m, int64_t col0, int64_t n_loc,
                       const double *params, int params_on_device);
/* bounds of this rank's entries (both NULL, or all -Inf/+Inf on EVERY rank = no bounds: optimize.jl:151); errors as
 * optimize.jl:144-148, :160-162.  Call on every rank (the "any finite bound" decision is all-reduced). */
int lfpsqp_large_set_bounds(lfpsqp_ctx *ctx, const double *xl_loc, const double *xu_loc);
int lfpsqp_large_solve(lfpsqp_ctx *ctx, const double *x0_loc, const lfpsqp_params *params, double *x_out_loc,
                       double *obj_hist, int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term,
                       lfpsqp_stats *stats);
/* the explicit-derivative core optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m, param) (src/optimize.jl:119-443)
 * for an ARBITRARY problem given by host callbacks: = lfpsqp_large_setup(LFPSQP_FAM_HOST) + set_bounds + large_solve.
 * lambda has length m.  The slack wrapper for d! (optimize.jl:13-71) stays on the host side, as in the reference. */
int lfpsqp_solve_host(lfpsqp_ctx *ctx, const lfpsqp_host_callbacks *cb, int64_t n, int64_t m, const double *x0,
                      const double *xl, const double *xu, const lfpsqp_params *params, double *x_out, double *obj_hist,
                      int64_t H, int64_t *obj_len, double *lambda, lfpsqp_term *term, lfpsqp_stats *stats);
/* unit-level ops mirroring the reference functions one to one (host buffers; outputs may be NULL):
 *   factor  : J = jac(x); G = J J' (m x m row-major, lower triangle valid), L = chol(G), Linv = L^-1   [ksvd!]
 *             *rank_deficient = 0, or the rank defect when the Cholesky pivot test failed (then L / Linv are undefined and the
 *             following project / projcg calls use the truncated pseudo-inverse, optimize.jl:297-302)
 *   project : v - J'(J J')^-1 J v and lambda = (J J')^-1 J v with the cached factor                    [kgemv! x2, optimize.jl:306-307, :333-343]
 *   projcg  : projcg! (src/projcg.jl:40-121) at x with multipliers lam on b = P(-grad f(x)), c = 0; status:
 *             1 converged, 2 negative curvature, 3 rg<=0, 4 iteration limit; ms = device time of the loop */
int lfpsqp_large_factor(lfpsqp_ctx *ctx, const double *x_loc, double *G_out, double *L_out, double *Linv_out,
                        int *rank_deficient, double *gram_ms);
int lfpsqp_large_project(lfpsqp_ctx *ctx, const double *v_loc, double *v_out_loc, double *lambda_out);
int lfpsqp_large_projcg(lfpsqp_ctx *ctx, const double *x_loc, const double *lam, double tol, int64_t maxit, int chunk,
                        double *sol_out_loc, int64_t *iters, double *nr, int *status, double *ms);

/*   projcg_general : projcg!(x, lambda, A, U, b, c; tol, maxit) (src/projcg.jl:40-121) in its general form (c != 0: x0 = U c, :55;
 *             test/test_cg.jl:10-28): A = the family's Lagrangian Hessian at (x, lam), U = the orthonormal Cholesky-QR basis
 *             J(x)' L^-T of range(J') (the reference's U up to an orthogonal change of basis), b (n_loc) and c (m) from the
 *             caller; lambda_out = U'(b - A sol) (:115-118; NaN after a negative-curvature exit).  Needs factor at x first. */
int lfpsqp_large_projcg_general(lfpsqp_ctx *ctx, const double *x_loc, const double *lam, const double *b_loc, const double *cvec,
                                double tol, int64_t maxit, double *sol_out_loc, double *lambda_out, int64_t *iters, double *nr,
                                int *status);

/*   retract : retract!(cval, xnew, c!, xtilde, x, method) (src/retractions.jl:75-177 NR [method 0] / :265-441 ProjPenalty
 *             [method 1]) with the factorisation at x_base, as armijo! calls it (src/linesearch.jl:52); flag as the reference
 *   pcg     : pcg!(mu, J, no_precondition, x=0, r=b, ...) (src/retractions.jl:179-246) with J = jac(x_point) */
int lfpsqp_large_retract(lfpsqp_ctx *ctx, int method, const double *x_base_loc, const double *xtilde_loc,
                         const lfpsqp_params *params, double *xnew_out_loc, double *cval_out, int *flag, int64_t *iters,
                         int64_t *pcg_iters);
int lfpsqp_large_pcg(lfpsqp_ctx *ctx, const double *x_point_loc, double mu, const double *b_loc, double tol, int64_t maxiter,
                     double *x_out_loc, double *r_out_loc, int *flag, int64_t *iters);

/* host wall-clock split (ms) of the last lfpsqp_large_solve: [factorisation (jac!, Gram, Cholesky, first projection),
 * projcg!, line search incl. retractions, total] */
int lfpsqp_large_phase_ms(lfpsqp_ctx *ctx, double *out4);

/* Unit-level bound embedding (src/inequality_helper.jl; y_retract! src/retractions.jl:451-500) on one instance; runs the
 * device code of the batched solver.  J: m x n row-major (== Jct column-major), may be NULL when m = 0.
 *  op 0 generate_initial_y! (:92-109)   in x (n)                          out xaug (2n)
 *  op 1 calculate_h! (:112-122)         in xaug (2n)                      out h (n)
 *  op 2 inequality_gradient! (:125-141) in xaug                           out [Dx | Dy | S] (3n)
 *  op 3 y_retract!                      in [xaug_base | xaug_trial] (4n)  out retracted trial (2n)
 *  op 4 bigA * v (:215-231)             in [xaug | v (n+m)]               out 2n
 *  op 5 bigA' * w (:254-271)            in [xaug | w (2n)]                out n+m
 *  op 6 d - Q Q'd, lambda, lambda_y (optimize.jl:316-317,:332; calculate_lambda_kkt! :286-308)
 *                                       in [xaug | d (2n)]                out [d_proj (2n) | lambda (m) | lambda_y (n)] */
int lfpsqp_ineq_op(lfpsqp_ctx *ctx, int op, int64_t n, int64_t m, const double *xl, const double *xu, const double *J,
                   const double *in, int64_t in_len, double *out, int64_t out_len);

/* Unit-level line search: armijo! (which = 0, src/linesearch.jl:32-89) / exact_linesearch! (which = 1, :107-339) on ONE
 * instance, called as the driver calls them (src/optimize.jl:396-420): g = grad f(x), fval = f(x), factorisation at x,
 * retraction by the driver's rule (m > 0: NR iff !do_project_retract else ProjPenalty; m = 0: YRetract with finite
 * bounds, else Euclidean).  x, d, xnew_out have the working length N (n, or 2n = [x | y] with finite bounds).
 * out6 = [newf, f_diff, step_diff, alpha, tot_iter1, tot_iter2] = the reference's return tuple after the flag.
 * Families: LFPSQP_FAM_BOXQUAD, LFPSQP_FAM_SIN.  Reference goldens: test/test_linesearch.jl:14-22 (alpha = 0.25), :24-32. */
int lfpsqp_linesearch(lfpsqp_ctx *ctx, int which, int family, int64_t n, int64_t m, const double *fam_params, const double *x,
                      const double *d, const double *xl, const double *xu, const lfpsqp_params *params, double *xnew_out,
                      double *out6, int *flag);
/* Unit-level augmented_hess_lag_vec! (src/inequality_helper.jl:144-158; test/test_inequalities.jl:157-177):
 * dest = [H(x, lam) src_x + 2 lam_y.q.src_x ; 2 lam_y.s.src_y] with H the family's hess_lag_vec! at xaug[1:n].
 * xaug, src, dest: 2n; lam: m; lamy: n.  Families: LFPSQP_FAM_BOXQUAD, LFPSQP_FAM_SIN. */
int lfpsqp_aug_hess_vec(lfpsqp_ctx *ctx, int family, int64_t n, int64_t m, const double *fam_params, const double *xl,
                        const double *xu, const double *xaug, const double *lam, const double *lamy, const double *src,
                        double *dest);

/* Communicator of the column-sharded large-n mode: one process per GPU, NCCL (bound with dlopen so the process shares
 * the libnccl.so.2 that e.g. torch.distributed loaded; nccl_lib_path may be NULL).  Rank 0 creates the 128-byte unique
 * id, the host program broadcasts it (any transport), every rank calls lfpsqp_comm_init BEFORE lfpsqp_large_setup. */
int lfpsqp_comm_unique_id(void *out128, const char *nccl_lib_path);
int lfpsqp_comm_init(lfpsqp_ctx *ctx, int rank, int world, const void *unique_id128, const char *nccl_lib_path);
int lfpsqp_comm_destroy(lfpsqp_ctx *ctx);
/* Peer-memory all-reduce for the small latency-bound messages of the large-n path (m-vectors, packed CG scalars): one
 * kernel per all-reduce that stores flags / loads partial sums directly in the peers' memory over NVLink (CUDA IPC),
 * summing in rank order (bitwise-identical result on every rank).  Each rank exports a 64-byte handle, the host
 * program all-gathers them (rank order) and every rank imports.  Without it NCCL carries these messages too. */
int lfpsqp_comm_ipc_export(lfpsqp_ctx *ctx, void *handle64_out);
int lfpsqp_comm_ipc_import(lfpsqp_ctx *ctx, const void *handles /* world x 64 bytes */);
int lfpsqp_comm_mode(lfpsqp_ctx *ctx); /* 0 single GPU, 1 NCCL only, 2 peer-memory kernels + NCCL (Gram) */

/* Roofline denominators that MEASURED_PEAKS.json does not carry: measured FP64 peak of this GPU in TFLOP/s.
 * which: 0 = DFMA (vector pipe), 1 = DMMA (mma.sync.m8n8k4.f64 tensor pipe). */
int lfpsqp_bench_fp64_peak(lfpsqp_ctx *ctx, int which, double *tflops);

#ifdef __cplusplus
}
#endif
#endif
