"""Large-n mode (one instance, dense m x n Jacobian, optionally column-sharded over GPUs) over the C ABI."""
import ctypes as C

import numpy as np

from . import _lib
from .api import LFPSQPParams, TerminationCondition, TerminationInfo, _family_of, _parse
from .families import DIAGQUAD, SPARSE_QCQP, SPARSE_QCQP_CSR, THOMSON

_SPARSE = (SPARSE_QCQP, SPARSE_QCQP_CSR)


class LargeProblem:
    """Binds one (sharded) problem to a Context: lfpsqp_large_setup, then solve / factor / project / projcg.

    Without bounds the working vectors of the unit-level calls (factor, project, projcg, pcg, retract) are this rank's n_loc
    entries of x.  With finite bounds (set_bounds) they are the 2 n_loc entries [x | y] of the embedding of
    src/inequality_helper.jl: factor returns the weighted Gram G_w = J diag(Dy^2) J' at that point, project returns the
    multipliers [lambda ; lambda_y] (m + n_loc entries), and projcg takes them in the same layout."""

    def __init__(self, fam, ctx=None, col0=0, n_loc=None, n_global=None, params_dev_ptr=None):
        self.ctx = ctx or _lib.default_context()
        self.fam = fam
        self.m = fam.m
        self.n_loc = fam.n if n_loc is None else n_loc
        self.n = fam.n if n_global is None else n_global
        if fam.id in _SPARSE and fam.p > 0:
            raise _lib.LFPSQPError("a sparse_qcqp with d(x) is solved by optimize_large, which adds the slack variables")
        if fam.id in _SPARSE and params_dev_ptr is None:
            pp, _keep = fam.large_args()
            on_dev = 0
        elif params_dev_ptr is not None:
            pp, on_dev = C.c_void_p(params_dev_ptr), 1
        else:
            pp, on_dev = _lib.ptr(fam.params), 0
        self.ctx.check(self.ctx.lib.lfpsqp_large_setup(self.ctx.h, fam.id, self.n, self.m, col0, self.n_loc, pp, on_dev))

    def set_bounds(self, xl, xu):
        """xl <= x <= xu for this rank's entries (None, None = no bounds): the 2n embedding of src/inequality_helper.jl"""
        xl = None if xl is None else np.ascontiguousarray(xl, dtype=np.float64)
        xu = None if xu is None else np.ascontiguousarray(xu, dtype=np.float64)
        if xl is not None and xu is not None and not (len(xl) == len(xu) == self.n_loc):
            raise _lib.LFPSQPError("xl, xu, and x0 must all be the same length")     # optimize.jl:144-148
        self.ctx.check(self.ctx.lib.lfpsqp_large_set_bounds(self.ctx.h, _lib.ptr(xl), _lib.ptr(xu)))

    @property
    def nv(self):
        """working length of the unit-level calls as the library holds it: n_loc, or 2 n_loc with the bound embedding
        (the library decides, after optimize.jl:151, and on every rank of a sharded problem alike)"""
        out = C.c_int64(0)
        self.ctx.check(self.ctx.lib.lfpsqp_large_working_length(self.ctx.h, C.byref(out)))
        return out.value

    def _working(self, v, what):
        v = np.ascontiguousarray(v, dtype=np.float64)
        nv = self.nv
        if v.shape != (nv,):
            raise _lib.LFPSQPError("%s must have the working length %d (%s), not %s"
                                   % (what, nv, "[x | y] with bounds" if nv != self.n_loc else "n_loc", v.shape))
        return v

    def solve(self, x0, param=None, history=None, return_stats=False, noise=None):
        """noise (beta > 0): (T, N_working_local) rows of the caller's randn! sequence (optimize.jl:264-273)"""
        param = param or LFPSQPParams()
        if noise is not None:
            noise = np.ascontiguousarray(noise, dtype=np.float64)
            self.ctx.check(self.ctx.lib.lfpsqp_ctx_set_noise(self.ctx.h, _lib.ptr(noise), noise.shape[0], noise.shape[1], 1))
        if history is None:   # every iterate's objective, as the reference returns (optimize.jl:250, :426)
            history = int(param.maxiter) + 1
        cp = param.to_c()
        x0 = np.ascontiguousarray(x0, dtype=np.float64)
        x = np.empty(self.n_loc); obj = np.full(history, np.nan); olen = np.zeros(1, dtype=np.int64)
        lam = np.zeros(max(self.m, 1)); term = np.zeros(1, dtype=_lib.TERM_DTYPE); stats = np.zeros(1, dtype=_lib.STATS_DTYPE)
        self.ctx.check(self.ctx.lib.lfpsqp_large_solve(self.ctx.h, _lib.ptr(x0), C.cast(C.pointer(cp), C.c_void_p), _lib.ptr(x),
                                                       _lib.ptr(obj), history, _lib.ptr(olen), _lib.ptr(lam), _lib.ptr(term),
                                                       _lib.ptr(stats)))
        if noise is not None:
            self.ctx.lib.lfpsqp_ctx_set_noise(self.ctx.h, None, 0, 0, 0)
        t = term[0]
        info = TerminationInfo(TerminationCondition(int(t["condition"])), float(t["f_diff"]), float(t["step_diff"]),
                               float(t["kkt_diff"]), int(t["iter"]))
        res = (x, obj[:min(int(olen[0]), history)].copy(), lam[:self.m], info)
        if return_stats:
            return res + ({k: int(stats[0][k]) for k in _lib.STATS_FIELDS}, int(t["status"]))
        return res

    def phase_ms(self):
        """[factorisation, projcg, line search, total] ms of the last solve()"""
        out = np.zeros(4)
        self.ctx.check(self.ctx.lib.lfpsqp_large_phase_ms(self.ctx.h, _lib.ptr(out)))
        return dict(factor=out[0], projcg=out[1], linesearch=out[2], total=out[3])

    def factor(self, x, want=("G", "L", "Linv")):
        m = self.m
        x = self._working(x, "x")
        G = np.zeros((m, m)) if "G" in want else None
        L = np.zeros((m, m)) if "L" in want else None
        Li = np.zeros((m, m)) if "Linv" in want else None
        rd = C.c_int(0); ms = C.c_double(0)
        self.ctx.check(self.ctx.lib.lfpsqp_large_factor(self.ctx.h, _lib.ptr(x), _lib.ptr(G), _lib.ptr(L), _lib.ptr(Li),
                                                        C.cast(C.pointer(rd), C.c_void_p), C.cast(C.pointer(ms), C.c_void_p)))
        return dict(G=G, L=L, Linv=Li, rank_deficient=rd.value, gram_ms=ms.value)

    def project(self, v):
        """-> (projected v, multipliers): lambda (m), or [lambda ; lambda_y] (m + n_loc) with bounds"""
        v = self._working(v, "v")
        nlam = self.m + (v.size - self.n_loc)
        out = np.empty_like(v); lam = np.zeros(max(nlam, 1))
        self.ctx.check(self.ctx.lib.lfpsqp_large_project(self.ctx.h, _lib.ptr(v), _lib.ptr(out), _lib.ptr(lam)))
        return out, lam[:nlam]

    def retract(self, method, x_base, xtilde, param=None):
        """retract! with method "nr" | "pp" -> (flag, xnew, cval, iters, pcg_iters)"""
        cp = (param or LFPSQPParams()).to_c()
        xb = self._working(x_base, "x_base"); xt = self._working(xtilde, "xtilde")
        xnew = np.empty_like(xb); cval = np.zeros(max(self.m, 1))
        fl = C.c_int(0); it = C.c_int64(0); pit = C.c_int64(0)
        self.ctx.check(self.ctx.lib.lfpsqp_large_retract(self.ctx.h, 0 if method == "nr" else 1, _lib.ptr(xb), _lib.ptr(xt),
                                                         C.cast(C.pointer(cp), C.c_void_p), _lib.ptr(xnew), _lib.ptr(cval),
                                                         C.cast(C.pointer(fl), C.c_void_p), C.cast(C.pointer(it), C.c_void_p),
                                                         C.cast(C.pointer(pit), C.c_void_p)))
        return fl.value, xnew, cval[:self.m], it.value, pit.value

    def pcg(self, x_point, mu, b, tol=1e-6, maxiter=100):
        """pcg! on (J'J + mu I) x = b with J = jac(x_point), or with bounds on (bigA bigA' + mu I) x = b -> (x, r, flag, iters)"""
        xp = self._working(x_point, "x_point"); b = self._working(b, "b")
        x = np.empty_like(xp); r = np.empty_like(xp); fl = C.c_int(0); it = C.c_int64(0)
        self.ctx.check(self.ctx.lib.lfpsqp_large_pcg(self.ctx.h, _lib.ptr(xp), mu, _lib.ptr(b), tol, maxiter, _lib.ptr(x), _lib.ptr(r),
                                                     C.cast(C.pointer(fl), C.c_void_p), C.cast(C.pointer(it), C.c_void_p)))
        return x, r, fl.value, it.value

    def projcg_general(self, x, lam, b, c, tol=1e-6, maxit=10000):
        """projcg!(x, lambda, A, U, b, c) (src/projcg.jl:40-121) with c != 0; needs factor(x) first.
        -> dict(sol, lam, iters, nr, status)"""
        f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
        x, lam, b, c = map(f64, (x, lam, b, c))
        sol = np.empty(self.n_loc); lout = np.zeros(max(self.m, 1))
        it = C.c_int64(0); nr = C.c_double(0); st = C.c_int(0)
        self.ctx.check(self.ctx.lib.lfpsqp_large_projcg_general(self.ctx.h, _lib.ptr(x), _lib.ptr(lam), _lib.ptr(b), _lib.ptr(c), tol, maxit,
                                                                _lib.ptr(sol), _lib.ptr(lout), C.cast(C.pointer(it), C.c_void_p),
                                                                C.cast(C.pointer(nr), C.c_void_p), C.cast(C.pointer(st), C.c_void_p)))
        return dict(sol=sol, lam=lout[:self.m], iters=it.value, nr=nr.value, status=st.value)

    def projcg(self, x, lam=None, tol=0.0, maxit=10, chunk=0, want_solution=True):
        """projcg! at x with multipliers lam (m, or [lambda ; lambda_y] of m + n_loc entries with bounds); needs factor(x) first"""
        x = self._working(x, "x")
        lam = None if lam is None else np.ascontiguousarray(lam, dtype=np.float64)
        if lam is not None and lam.shape != (self.m + x.size - self.n_loc,):
            raise _lib.LFPSQPError("lam must have %d entries, not %s" % (self.m + x.size - self.n_loc, lam.shape))
        sol = np.empty_like(x) if want_solution else None
        it = C.c_int64(0); nr = C.c_double(0); st = C.c_int(0); ms = C.c_double(0)
        self.ctx.check(self.ctx.lib.lfpsqp_large_projcg(self.ctx.h, _lib.ptr(x), _lib.ptr(lam), tol, maxit, chunk, _lib.ptr(sol),
                                                        C.cast(C.pointer(it), C.c_void_p), C.cast(C.pointer(nr), C.c_void_p),
                                                        C.cast(C.pointer(st), C.c_void_p), C.cast(C.pointer(ms), C.c_void_p)))
        return dict(sol=sol, iters=it.value, nr=nr.value, status=st.value, ms=ms.value)


def linesearch(which, fam, x, d, xl=None, xu=None, param=None, ctx=None):
    """armijo! / exact_linesearch! (src/linesearch.jl:32-89, :107-339) on one instance, as the driver calls them.
    which: "armijo" | "exact".  x, d: working length (n, or 2n = [x | y] with finite bounds).
    -> (flag, tot_iter1, tot_iter2, newf, f_diff, step_diff, alpha, xnew): the reference's return tuple + xnew."""
    ctx = ctx or _lib.default_context()
    cp = (param or LFPSQPParams()).to_c()
    x = np.ascontiguousarray(x, dtype=np.float64); d = np.ascontiguousarray(d, dtype=np.float64)
    xl = None if xl is None else np.ascontiguousarray(xl, dtype=np.float64)
    xu = None if xu is None else np.ascontiguousarray(xu, dtype=np.float64)
    fp = np.ascontiguousarray(fam.params, dtype=np.float64).ravel()
    xnew = np.empty_like(x); out6 = np.zeros(6); fl = C.c_int(0)
    ctx.check(ctx.lib.lfpsqp_linesearch(ctx.h, 0 if which == "armijo" else 1, fam.id, fam.n, fam.m, _lib.ptr(fp), _lib.ptr(x),
                                        _lib.ptr(d), _lib.ptr(xl), _lib.ptr(xu), C.cast(C.pointer(cp), C.c_void_p), _lib.ptr(xnew),
                                        _lib.ptr(out6), C.cast(C.pointer(fl), C.c_void_p)))
    return fl.value, int(out6[4]), int(out6[5]), out6[0], out6[1], out6[2], out6[3], xnew


def aug_hess_vec(fam, xl, xu, xaug, lam, lamy, src, ctx=None):
    """augmented_hess_lag_vec! (src/inequality_helper.jl:144-158) on the device: -> dest (2n)."""
    ctx = ctx or _lib.default_context()
    f64 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float64)
    xl, xu, xaug, lam, lamy, src = map(f64, (xl, xu, xaug, lam, lamy, src))
    fp = np.ascontiguousarray(fam.params, dtype=np.float64).ravel()
    dest = np.zeros(2 * fam.n)
    ctx.check(ctx.lib.lfpsqp_aug_hess_vec(ctx.h, fam.id, fam.n, fam.m, _lib.ptr(fp), _lib.ptr(xl), _lib.ptr(xu), _lib.ptr(xaug),
                                          _lib.ptr(lam), _lib.ptr(lamy), _lib.ptr(src), _lib.ptr(dest)))
    return dest


def ineq_op(op, xl, xu, inp, J=None, ctx=None):
    """Unit-level bound-embedding ops on the device (lfpsqp_ineq_op): op in {"initial_y", "h", "gradient", "y_retract",
    "bigA", "bigAt", "project"}.  J: (m, n) row-major (= Jct', src/optimize.jl:190)."""
    ctx = ctx or _lib.default_context()
    code = dict(initial_y=0, h=1, gradient=2, y_retract=3, bigA=4, bigAt=5, project=6)[op]
    xl = np.ascontiguousarray(xl, dtype=np.float64); xu = np.ascontiguousarray(xu, dtype=np.float64)
    n = len(xl); m = 0 if J is None else J.shape[0]
    Jc = None if J is None else np.ascontiguousarray(J, dtype=np.float64)
    inp = np.ascontiguousarray(inp, dtype=np.float64)
    olen = [2 * n, n, 3 * n, 2 * n, 2 * n, n + m, 3 * n + m][code]
    out = np.zeros(olen)
    ctx.check(ctx.lib.lfpsqp_ineq_op(ctx.h, code, n, m, _lib.ptr(xl), _lib.ptr(xu), _lib.ptr(Jc), _lib.ptr(inp), inp.size,
                                     _lib.ptr(out), olen))
    return out


def make_diagquad(n, m, seed=0, cond=1e4, dtype=np.float64):
    """BASELINE config C5 (definition pinned in SURVEY.md 8d / DESIGN.md): Q, A ~ N(0,1)/sqrt(n), x0 ~ N(0,1),
    b such that c(x0) = 0, f = 1/2 (x-xt)' diag(w) (x-xt) with w log-uniform in [1, cond]."""
    rng = np.random.Generator(np.random.Philox(key=seed))
    Q = rng.standard_normal((m, n)) / np.sqrt(n); A = rng.standard_normal((m, n)) / np.sqrt(n)
    x0 = rng.standard_normal(n); xt = rng.standard_normal(n)
    w = np.exp(rng.uniform(0.0, np.log(cond), n))
    b = 0.5 * Q @ (x0 * x0) + A @ x0
    return Q, A, b, xt, w, x0


def optimize_large(*args, ctx=None, history=None, return_stats=False, noise=None):
    """optimize(...) for ONE large instance of a large-n device family (diagquad, thomson, sparse_qcqp) on one GPU, with the
    reference's method shapes (optimize.jl:13, :83, :88, :107, :112) -> (x, obj_values, λ_kkt, term_info).

    With d(x) (sparse_qcqp only) the slack wrapper of optimize.jl:13-71 is built as data (SparseQCQPFamily.slack_embedding):
    variables [x ; s], equalities [c(x) ; d(x) - s], bounds [xl ; dl] <= [x ; s] <= [xu ; du]; λ then has m + p entries
    (optimize.jl:67-70).  noise (beta > 0): (T, N_working) rows of the caller's randn! sequence, N_working = 2 (n + p) with
    bounds, else n."""
    f, c, d, dl, du, x0, xl, xu, m, p, param = _parse(args)
    fam = _family_of(f, c, d)
    if fam.id not in (DIAGQUAD, THOMSON) + _SPARSE:
        raise _lib.LFPSQPError("optimize_large takes a large-n device family (diagquad, thomson, sparse_qcqp); %r is not one"
                               % fam)
    if d is None or p == 0:                                                              # optimize.jl:15-17
        p = 0
    if c is None and m != 0:
        raise _lib.LFPSQPError("c! is nothing but m > 0")
    x0 = np.ascontiguousarray(x0, dtype=np.float64)
    if x0.ndim != 1 or (x0.size, m, p) != (fam.n, fam.m, fam.p if p > 0 else 0):
        raise _lib.LFPSQPError("sizes (n=%d, m=%d, p=%d) do not match the family %r" % (x0.size, m, p, fam))
    if (xl is None) != (xu is None):
        raise _lib.LFPSQPError("xl and xu must both be given or both be nothing")
    if xl is not None and not (len(xl) == len(xu) == x0.size):
        raise _lib.LFPSQPError("xl, xu, and x0 must all be the same length")             # optimize.jl:144-148
    param = param or LFPSQPParams()
    if history is None:   # every iterate's objective, as the reference returns (optimize.jl:250, :426)
        history = int(param.maxiter) + 1
    if p > 0:
        if fam.id not in _SPARSE:
            raise _lib.LFPSQPError("d(x) in large-n mode needs a sparse_qcqp family (its slack variables are data)")
        prob_fam, x0w, xl, xu = fam.slack_embedding(x0, xl, xu, dl, du)
    else:
        prob_fam, x0w = fam, x0
        if fam.id in _SPARSE and fam.p > 0:   # d! not passed (or p = 0): the equalities alone
            prob_fam = fam.equalities()
    prob = LargeProblem(prob_fam, ctx=ctx)
    prob.set_bounds(xl, xu)
    out = prob.solve(x0w, param, history=history, return_stats=return_stats, noise=noise)
    if out[3].iter == param.maxiter:
        import warnings
        warnings.warn("Maximum # of outer iterations reached")                           # optimize.jl:438-440
    return (out[0][:fam.n],) + tuple(out[1:])                                            # :67-70 (lambda untruncated)
