"""Host mirror of the reference's public API (src/optimize.jl:13-114, src/LFPSQP.jl:27-81)."""
import ctypes as C
import enum
from typing import NamedTuple

import numpy as np

from . import _lib
from .families import QCQP, SPARSE_QCQP, SPARSE_QCQP_CSR, DeviceCallback

# LinesearchOption / DisplayOption (src/LFPSQP.jl:27-35)
armijo, exact = 0, 1
off, iter_ = 0, 1


class TerminationCondition(enum.IntEnum):  # src/LFPSQP.jl:37-43
    f_tol = 0
    x_tol = 1
    kkt_tol = 2
    max_iter = 3
    armijo_error = 4


class TerminationInfo(NamedTuple):  # src/LFPSQP.jl:45-54
    condition: TerminationCondition
    f_diff: float
    step_diff: float
    kkt_diff: float
    iter: int

    def __str__(self):
        return ("TerminationInfo:\ncondition = %s\n       Δf = %r\n   ||Δx|| = %r\n||P(∇f)|| = %r\n    iters = %d"
                % (self.condition.name, self.f_diff, self.step_diff, self.kkt_diff, self.iter))


_GREEK = {"α": "alpha", "β": "beta", "t_β": "t_beta", "σ": "sigma", "ϵ_c": "eps_c", "ϵ_f": "eps_f", "ϵ_x": "eps_x",
          "ϵ_kkt": "eps_kkt", "ϵ_rank": "eps_rank", "μ0": "mu0", "tn_κ": "tn_kappa"}
# Python NFKC-normalises identifiers: the reference's lunate epsilon (U+03F5) arrives as U+03B5
_GREEK.update({k.replace("\u03f5", "\u03b5"): v for k, v in list(_GREEK.items()) if "\u03f5" in k})


class LFPSQPParams:
    """Keyword struct with the reference's fields and defaults (src/LFPSQP.jl:57-81).  Both the reference's Greek
    field names (α, ϵ_c, μ0, tn_κ ...) and ASCII spellings (alpha, eps_c, mu0, tn_kappa ...) are accepted."""

    _defaults = dict(alpha=1.0, beta=0.0, t_beta=0, s=0.5, sigma=1e-4, eps_c=1e-6, eps_f=1e-6, eps_x=0.0,
                     eps_kkt=1e-6, eps_rank=1e-10, maxiter=10000, maxiter_retract=100, maxiter_pcg=100, mu0=1e-2,
                     disable_linesearch=False, do_project_retract=True, disp=iter_, callback=None,
                     callback_period=100, linesearch=armijo, do_newton=True, tn_maxiter=10000, tn_kappa=0.5)

    def __init__(self, **kw):
        vals = dict(self._defaults)
        for k, v in kw.items():
            k = _GREEK.get(k, k)
            if k not in vals:
                raise TypeError("LFPSQPParams has no field %r" % k)
            vals[k] = v
        self.__dict__.update(vals)

    def __getattr__(self, k):  # Greek aliases
        if k in _GREEK:
            return self.__dict__[_GREEK[k]]
        raise AttributeError(k)

    def to_c(self):
        if self.callback is not None:
            raise _lib.LFPSQPError("param.callback (optimize.jl:432-434) needs the host-callback form "
                                    "optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m, param); registered device "
                                    "families run whole solves on the GPU without returning to the host")
        p = _lib.CParams()
        for name, _ in _lib.CParams._fields_:
            if name == "_pad":
                continue
            v = self.__dict__[name]
            setattr(p, name, int(v) if isinstance(v, (bool, np.bool_)) else v)
        return p


def _family_of(f, c, d):
    if not isinstance(f, DeviceCallback) or f.role != "f":
        raise TypeError("f must be the .f handle of a registered device family (lfpsqp.jl_b200.families); "
                        "host closures cannot run on the GPU")
    fam = f.family
    for cb, role in ((c, "c"), (d, "d")):
        if cb is not None and (not isinstance(cb, DeviceCallback) or cb.family is not fam or cb.role != role):
            raise TypeError("%s! must be the .%s handle of the same family as f" % (role, role))
    return fam


def _parse(args):
    """Resolve the reference's method family by shape (optimize.jl:13, :83, :88, :107, :112)."""
    args = list(args)
    param = args.pop() if args and isinstance(args[-1], LFPSQPParams) else LFPSQPParams()
    f = args[0]
    na = len(args)
    dl = du = None
    if na == 2:       # optimize(f, x0)
        c = d = None; x0 = args[1]; xl = xu = None; m = p = 0
    elif na == 4:     # optimize(f, c!, x0, m)
        c, x0, m = args[1], args[2], args[3]; d = None; xl = xu = None; p = 0
    elif na == 6:     # optimize(f, c!, x0, xl, xu, m)
        c, x0, xl, xu, m = args[1:6]; d = None; p = 0
    elif na == 8:     # optimize(f, c!, d!, x0, xl, xu, m, p)
        c, d, x0, xl, xu, m, p = args[1:8]
    elif na == 10:    # optimize(f, c!, d!, dl, du, x0, xl, xu, m, p)
        c, d, dl, du, x0, xl, xu, m, p = args[1:10]
    else:
        raise TypeError("no method matching optimize with %d positional arguments" % na)
    return f, c, d, dl, du, x0, xl, xu, int(m), int(p), param


def optimize_batched(*args, ctx=None, history=64, return_stats=False, noise=None):
    """B independent instances in lockstep on one GPU.  Same positional shapes as `optimize`, with x0 of shape
    (B, n) and per-instance family parameters of shape (B, P).  Returns (x (B,n), obj_values (B,H) NaN-padded,
    obj_len (B,), lambda (B,m+p), term (B,) structured array[, stats])."""
    f, c, d, dl, du, x0, xl, xu, m, p, param = _parse(args)
    fam = _family_of(f, c, d)
    if fam.id in (SPARSE_QCQP, SPARSE_QCQP_CSR):
        raise _lib.LFPSQPError("sparse_qcqp is a large-n family (one large instance on one GPU): call optimize_large")
    if d is None or p == 0:   # optimize.jl:15-17
        p = 0
    if c is None:
        if m != 0 and fam.m != 0:
            raise _lib.LFPSQPError("c! is nothing but m > 0")
    x0 = np.ascontiguousarray(x0, dtype=np.float64)
    if x0.ndim != 2:
        raise _lib.LFPSQPError("optimize_batched: x0 must be (B, n)")
    B, n = x0.shape
    if (n, m, p) != (fam.n, fam.m, fam.p):
        raise _lib.LFPSQPError("sizes (n=%d, m=%d, p=%d) do not match the family %r" % (n, m, p, fam))
    if p > 0:
        if dl is not None or du is not None:
            dl = np.asarray(dl, float); du = np.asarray(du, float)
            if not (len(dl) == len(du) == p):
                raise _lib.LFPSQPError("Bound vectors dl and du must be of size p")   # optimize.jl:19-21
            if not (np.all(np.isneginf(dl)) and np.all(du == 0.0)):
                raise _lib.LFPSQPError("only d(x) <= 0 (dl=-Inf, du=0; optimize.jl:83-85) is on the device path")
        if xl is None: xl = -np.inf * np.ones(n)
        if xu is None: xu = np.inf * np.ones(n)
    if (xl is None) != (xu is None):
        raise _lib.LFPSQPError("xl and xu must both be given or both be nothing")
    if xl is not None:
        xl = np.ascontiguousarray(xl, dtype=np.float64); xu = np.ascontiguousarray(xu, dtype=np.float64)
        if not (len(xl) == len(xu) == n):
            raise _lib.LFPSQPError("xl, xu, and x0 must all be the same length")      # optimize.jl:144-148
    ctx = ctx or _lib.default_context()
    cp = param.to_c()
    fp, stride, keep = fam.batched_args(B)
    H = int(history)
    x = np.empty((B, n)); obj = np.empty((B, H)); olen = np.zeros(B, dtype=np.int64)
    lam = np.zeros((B, m + p)); term = np.zeros(B, dtype=_lib.TERM_DTYPE)
    stats = np.zeros(B, dtype=_lib.STATS_DTYPE) if return_stats else None
    if noise is not None:   # beta > 0: the caller's randn! rows, (B, T, N_working) (optimize.jl:264-273)
        noise = np.ascontiguousarray(noise, dtype=np.float64)
        if noise.ndim != 3 or noise.shape[0] != B:
            raise _lib.LFPSQPError("noise must have shape (B, T, N_working)")
        ctx.check(ctx.lib.lfpsqp_ctx_set_noise(ctx.h, _lib.ptr(noise), noise.shape[1], noise.shape[2], B))
    rc = ctx.lib.lfpsqp_solve_batched(ctx.h, fam.id, n, m, p, B, fp, stride, _lib.ptr(x0), _lib.ptr(xl),
                                      _lib.ptr(xu), C.cast(C.pointer(cp), C.c_void_p), _lib.ptr(x), _lib.ptr(obj), H,
                                      _lib.ptr(olen), _lib.ptr(lam), _lib.ptr(term), _lib.ptr(stats))
    del keep
    if noise is not None:
        ctx.lib.lfpsqp_ctx_set_noise(ctx.h, None, 0, 0, 0)
    ctx.check(rc)
    if B and int(olen.max()) > H:
        import warnings
        warnings.warn("obj_values holds the first %d objective values per instance; the longest history has %d (the reference returns "
                      "every iterate's objective, optimize.jl:426): pass history=maxiter+1 to keep them all" % (H, int(olen.max())))
    if return_stats:
        return x, obj, olen, lam, term, stats
    return x, obj, olen, lam, term


def optimize(*args, ctx=None, history=None, return_stats=False, noise=None):
    """optimize(f, x0[, param]) / (f, c!, x0, m[, param]) / (f, c!, x0, xl, xu, m[, param]) /
    (f, c!, d!, x0, xl, xu, m, p[, param]) / (f, c!, d!, dl, du, x0, xl, xu, m, p[, param])
    -> (x, obj_values, λ_kkt, term_info), as src/optimize.jl:442."""
    a = list(args)
    param = a.pop() if a and isinstance(a[-1], LFPSQPParams) else None
    if history is None:     # every iterate's objective, as the reference returns (optimize.jl:250, :426)
        history = int((param or LFPSQPParams()).maxiter) + 1
    if len(a) == 9 and callable(a[0]) and not isinstance(a[0], DeviceCallback):
        # the explicit-derivative core optimize(f, grad!, c!, jac!, hess_lag_vec!, x0, xl, xu, m, param) (optimize.jl:119)
        # with host callables: generic problems, linear algebra on the device (host.py)
        from .host import optimize_explicit
        return optimize_explicit(*a, param, ctx=ctx, history=history, return_stats=return_stats)
    # locate x0 in the positional list and add the batch axis
    idx = {2: 1, 4: 2, 6: 2, 8: 3, 10: 5}.get(len(a))
    if idx is None:
        raise TypeError("no method matching optimize with %d positional arguments" % len(a))
    if isinstance(a[0], DeviceCallback) and a[0].family.id == QCQP and a[0].family.batched_params:
        raise _lib.LFPSQPError("optimize solves one instance: give every qcqp array at its own shape (no batch axis), "
                               "or call optimize_batched")
    a[idx] = np.asarray(a[idx], dtype=np.float64)[None, :]
    if param is not None:
        a.append(param)
    out = optimize_batched(*a, ctx=ctx, history=history, return_stats=return_stats,
                           noise=None if noise is None else np.asarray(noise, dtype=np.float64)[None])
    x, obj, olen, lam, term = out[:5]
    t = term[0]
    info = TerminationInfo(TerminationCondition(int(t["condition"])), float(t["f_diff"]), float(t["step_diff"]),
                           float(t["kkt_diff"]), int(t["iter"]))
    if int(t["iter"]) == (param or LFPSQPParams()).maxiter:
        import warnings
        warnings.warn("Maximum # of outer iterations reached")     # optimize.jl:438-440
    res = (x[0], obj[0, :min(int(olen[0]), obj.shape[1])].copy(), lam[0], info)
    if return_stats:
        return res + ({k: int(out[5][0][k]) for k in _lib.STATS_FIELDS}, int(t["status"]))
    return res
