"""Registered device problem families.

Julia closures cannot run on the GPU, so the `f`, `c!`, `d!` arguments of `optimize` are handles onto device code
compiled into liblfpsqp_b200.so (family id + parameter blob), implementing the callback contract of
src/autodiff_generators.jl (grad! :7-9, jac! :40-42, hess_lag_vec! :80-104) analytically.

    fam = families.readme_inequality(coeff)
    x, obj_values, lam, term_info = optimize(fam.f, None, fam.d, x0, xl, xu, 0, 1)
"""
import ctypes as C

import numpy as np

from . import _lib

ROSENBROCK, README_EQ, README_INEQ, THOMSON, DIAGQUAD, SIN, BOXQUAD = range(7)
QCQP = 101


class DeviceCallback:
    """A handle onto one role ('f', 'c', 'd') of a registered device family."""

    def __init__(self, family, role):
        self.family = family
        self.role = role

    def __repr__(self):
        return "<device %s of %r>" % (self.role, self.family)


class Family:
    def __init__(self, fam_id, name, n, m, p, params=None, batched_params=False):
        self.id = fam_id
        self.name = name
        self.n, self.m, self.p = n, m, p
        # params: (P,) shared blob or (B, P) per-instance blobs
        self.params = None if params is None else np.ascontiguousarray(params, dtype=np.float64)
        self.batched_params = batched_params
        self.f = DeviceCallback(self, "f")
        self.c = DeviceCallback(self, "c") if m > 0 else None
        self.d = DeviceCallback(self, "d") if p > 0 else None

    def __repr__(self):
        return "Family(%s, n=%d, m=%d, p=%d)" % (self.name, self.n, self.m, self.p)

    def batched_args(self, B):
        """(fam_params pointer, fam_stride, object to keep alive during the call) of lfpsqp_solve_batched for B instances."""
        fp = self.params
        stride = 0
        if fp is not None and self.batched_params:
            if fp.shape[0] != B:
                raise _lib.LFPSQPError("per-instance family parameters must have B rows")
            stride = fp.shape[1]
        return _lib.ptr(fp), stride, fp


class QCQPFamily(Family):
    """Dense QCQP given by data (lfpsqp_qcqp); see qcqp()."""

    def __init__(self, arrays, n, m, p, B):
        super().__init__(QCQP, "qcqp", n, m, p, batched_params=B is not None)
        self.arrays = arrays      # name -> (C-contiguous float64 array, per_instance)
        self.B = B                # batch size of the per-instance arrays, None when every array is shared

    def batched_args(self, B):
        if self.B is not None and self.B != B:
            raise _lib.LFPSQPError("qcqp: per-instance arrays have %d instances, the batch has %d" % (self.B, B))
        desc = _lib.CQcqp()
        for name, (a, per_instance) in self.arrays.items():
            setattr(desc, name, a.ctypes.data)
            setattr(desc, name + "_stride", a[0].size if per_instance else 0)
        return C.cast(C.pointer(desc), C.c_void_p), 0, (desc, self.arrays)


def rosenbrock():
    """README.md:18-22: f(x) = (1-x1)^2 + 100 (x2 - x1^2)^2."""
    return Family(ROSENBROCK, "rosenbrock", 2, 0, 0)


def readme_equality(n=50):
    """README.md:41-54: f = dot(x,x), c = x[1] - 0.75."""
    return Family(README_EQ, "readme_eq", n, 1, 0)


def readme_inequality(coeff):
    """README.md:57-76: f = dot(coeff, x), d = dot(x,x) - 1 <= 0.  coeff: (n,) or (B, n) for a batch."""
    coeff = np.asarray(coeff, dtype=np.float64)
    return Family(README_INEQ, "readme_ineq", coeff.shape[-1], 0, 1, coeff, batched_params=coeff.ndim == 2)


def thomson(npoints):
    """f = sum_{i<j} 1/|x_i - x_j|, c_i = |x_i|^2 - 1; n = 3*npoints, m = npoints."""
    return Family(THOMSON, "thomson", 3 * npoints, npoints, 0)


def diagquad(Q, A, b, xt, w):
    """c_i = 1/2 sum_j Q_ij x_j^2 + A_i.x - b_i ; f = 1/2 sum_j w_j (x_j - xt_j)^2.  Q, A: (m, n)."""
    Q = np.asarray(Q, dtype=np.float64); A = np.asarray(A, dtype=np.float64)
    m, n = Q.shape
    blob = np.concatenate([Q.ravel(), A.ravel(), np.asarray(b, float).ravel(), np.asarray(xt, float).ravel(),
                           np.asarray(w, float).ravel()])
    return Family(DIAGQUAD, "diagquad", n, m, 0, blob)


def sin_system(n, m, t=None):
    """test/test_retractions.jl:34-54: c_i = x[2i] - sin(x[2i-1]); objective 1/2 |x - t|^2."""
    t = np.zeros(n) if t is None else np.asarray(t, dtype=np.float64)
    return Family(SIN, "sin", n, m, 0, t, batched_params=t.ndim == 2)


def boxquad(t, a=None, b=0.0):
    """f = |x - t|^2 with an optional linear equality a.x = b (used with bounds xl <= x <= xu)."""
    t = np.asarray(t, dtype=np.float64)
    n = t.shape[-1]
    m = 0 if a is None else 1
    av = np.zeros(n) if a is None else np.asarray(a, dtype=np.float64)
    if t.ndim == 2:
        B = t.shape[0]
        blob = np.concatenate([t, np.broadcast_to(av, (B, n)), np.full((B, 1), float(b))], axis=1)
        return Family(BOXQUAD, "boxquad", n, m, 0, blob, batched_params=True)
    return Family(BOXQUAD, "boxquad", n, m, 0, np.concatenate([t, av, [float(b)]]))


# own shape of each lfpsqp_qcqp array, in dimensions named n (variables), m (equalities), p (inequalities)
_QCQP_SHAPES = dict(P="nn", q="n", r="", Qc="mnn", Ac="mn", bc="m", Qd="pnn", Ad="pn", bd="p")


def qcqp(P=None, q=None, r=None, Qc=None, Ac=None, bc=None, Qd=None, Ad=None, bd=None):
    """Dense quadratically constrained quadratic program (batched mode):

        f(x)   = 1/2 x'P x + q.x + r
        c_i(x) = 1/2 x'Qc[i] x + Ac[i].x - bc[i] = 0      i < m
        d_k(x) = 1/2 x'Qd[k] x + Ad[k].x - bd[k] <= 0     k < p

    Each array is given at its own shape -- P (n, n), q (n,), r scalar, Qc (m, n, n), Ac (m, n), bc (m,), Qd (p, n, n),
    Ad (p, n), bd (p,) -- and is then shared by the batch, or with a leading batch axis B for one copy per instance.
    None is all zero.  n, m and p are inferred from the shapes.  Matrices are symmetrised as (M + M')/2, which leaves
    the quadratic forms unchanged (and every entry, when M is symmetric already).

        fam = families.qcqp(P=A, Qc=np.eye(n)[None], bc=[0.5])        # Rayleigh quotient on the unit sphere
        x, obj, olen, lam, term = optimize_batched(fam.f, fam.c, x0, fam.m)
    """
    given = {k: v for k, v in dict(P=P, q=q, r=r, Qc=Qc, Ac=Ac, bc=bc, Qd=Qd, Ad=Ad, bd=bd).items() if v is not None}
    dims, B, arrays = {}, None, {}
    for name, a in given.items():
        a = np.asarray(a, dtype=np.float64)
        own = _QCQP_SHAPES[name]
        if a.ndim == len(own):
            per_instance = False
        elif a.ndim == len(own) + 1:
            per_instance = True
            if B is not None and a.shape[0] != B:
                raise _lib.LFPSQPError("qcqp: %s has %d instances, another array has %d" % (name, a.shape[0], B))
            B = a.shape[0]
        else:
            raise _lib.LFPSQPError("qcqp: %s must have shape (%s) or (B, %s), got %s"
                                   % (name, ", ".join(own), ", ".join(own), a.shape))
        for d, size in zip(own, a.shape[1:] if per_instance else a.shape):
            if dims.setdefault(d, size) != size:
                raise _lib.LFPSQPError("qcqp: %s gives %s = %d, another array gives %d" % (name, d, size, dims[d]))
        if own.endswith("nn"):
            a = 0.5 * (a + np.swapaxes(a, -1, -2))
        arrays[name] = (np.ascontiguousarray(a), per_instance)
    if "n" not in dims:
        raise _lib.LFPSQPError("qcqp: n is unknown (give P, q, Qc, Ac, Qd or Ad)")
    n, m, p = dims["n"], dims.get("m", 0), dims.get("p", 0)
    if n < 1:
        raise _lib.LFPSQPError("qcqp: n must be at least 1")
    if m > 0 and "Qc" not in arrays and "Ac" not in arrays:
        raise _lib.LFPSQPError("qcqp: m = %d equalities need Qc or Ac" % m)
    if p > 0 and "Qd" not in arrays and "Ad" not in arrays:
        raise _lib.LFPSQPError("qcqp: p = %d inequalities need Qd or Ad" % p)
    for name in [k for k in arrays if _QCQP_SHAPES[k][:1] in ("m", "p") and dims[_QCQP_SHAPES[k][0]] == 0]:
        del arrays[name]      # empty constraint blocks: nothing to pass
    return QCQPFamily(arrays, n, m, p, B)
