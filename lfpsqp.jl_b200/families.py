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
SPARSE_QCQP = 102
SPARSE_QCQP_CSR = 103   # the same problem with its Jacobian kept sparse on the device (jacobian="csr")
_JACOBIAN_IDS = {"dense": SPARSE_QCQP, "csr": SPARSE_QCQP_CSR}


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


def _coo_of(M, name):
    """(row, col, val) of a matrix given as anything with .tocoo() (scipy.sparse) or as a dense 2-D array, and its shape"""
    if hasattr(M, "tocoo"):
        c = M.tocoo()
        r, k, v, shape = c.row, c.col, c.data, tuple(c.shape)
    else:
        a = np.asarray(M, dtype=np.float64)
        if a.ndim != 2:
            raise _lib.LFPSQPError("sparse_qcqp: %s must be a matrix (2-D array or scipy.sparse), got shape %s" % (name, a.shape))
        r, k = np.nonzero(a)
        v, shape = a[r, k], a.shape
    return np.asarray(r, np.int64), np.asarray(k, np.int64), np.asarray(v, np.float64), shape


def _summed(r, k, v, ncols):
    """duplicates summed (in input order), entries sorted by (row, col), exact zeros dropped"""
    key, inv = np.unique(r * ncols + k, return_inverse=True)
    s = np.bincount(inv.ravel(), weights=v, minlength=key.size)
    nz = s != 0.0
    return key[nz] // ncols, key[nz] % ncols, s[nz]


def _symmetrised(r, k, v, n):
    """(M + M')/2: each entry becomes 1/2 (M[r, c] + M[c, r]), a sum of two terms, so the result is exactly symmetric"""
    r, k, v = _summed(r, k, v, n)
    return _summed(np.concatenate([r, k]), np.concatenate([k, r]), 0.5 * np.concatenate([v, v]), n)


def _coo_matvec(r, k, v, x, nrows):
    return np.bincount(r, weights=v * x[k], minlength=nrows)


class SparseQCQPFamily(Family):
    """Sparse QCQP given by data (lfpsqp_sparse_qcqp, large-n mode); see sparse_qcqp().  Holds the canonical coordinate
    lists: P, Ac, Ad as (row, col, val); Qc, Qd as (mat, row, col, val), sorted, duplicates summed, symmetric.
    jacobian: the storage of J on the device, "dense" (family SPARSE_QCQP) or "csr" (SPARSE_QCQP_CSR)."""

    def __init__(self, n, m, p, P, q, r, Qc, Ac, bc, Qd, Ad, bd, jacobian="dense"):
        if jacobian not in _JACOBIAN_IDS:
            raise _lib.LFPSQPError('sparse_qcqp: jacobian must be "dense" or "csr", got %r' % (jacobian,))
        super().__init__(_JACOBIAN_IDS[jacobian], "sparse_qcqp", n, m, p)
        self.jacobian = jacobian
        self.P, self.q, self.r, self.Qc, self.Ac, self.bc = P, q, float(r), Qc, Ac, bc
        self.Qd, self.Ad, self.bd = Qd, Ad, bd

    def large_args(self):
        """(descriptor pointer for lfpsqp_large_setup, object to keep alive during the call) of the equalities c = 0"""
        def coo(t, stacked):
            c = _lib.CCoo()
            c.nnz = t[-1].size
            if stacked:
                c.mat = t[0].ctypes.data
            c.row, c.col, c.val = (a.ctypes.data for a in t[-3:])
            return c
        desc = _lib.CSparseQcqp()
        desc.P, desc.Qc, desc.Ac = coo(self.P, False), coo(self.Qc, True), coo(self.Ac, False)
        desc.q, desc.r, desc.bc = self.q.ctypes.data, self.r, self.bc.ctypes.data
        keep = (desc, self.P, self.Qc, self.Ac, self.q, self.bc)
        return C.cast(C.pointer(desc), C.c_void_p), keep

    def slack_embedding(self, x0, xl=None, xu=None, dl=None, du=None):
        """The slack wrapper of src/optimize.jl:13-71 written as data: variables [x ; s] with s0 = d(x0), equalities
        [c(x) ; d(x) - s] (Ad_k gains -1 in column n + k), bounds [xl ; dl] <= [x ; s] <= [xu ; du] (dl = -Inf, du = 0
        by default, optimize.jl:83-85).  -> (family with p = 0, x0_aug, xl_aug, xu_aug)"""
        n, m, p = self.n, self.m, self.p
        dl = -np.inf * np.ones(p) if dl is None else np.asarray(dl, dtype=np.float64).ravel()
        du = np.zeros(p) if du is None else np.asarray(du, dtype=np.float64).ravel()
        if not (len(dl) == len(du) == p):
            raise _lib.LFPSQPError("Bound vectors dl and du must be of size p")                 # optimize.jl:19-21
        x0 = np.asarray(x0, dtype=np.float64)
        xl = -np.inf * np.ones(n) if xl is None else np.asarray(xl, dtype=np.float64)
        xu = np.inf * np.ones(n) if xu is None else np.asarray(xu, dtype=np.float64)
        cat = np.concatenate
        Qc = tuple(cat([a, b]) for a, b in zip(self.Qc, (self.Qd[0] + m,) + self.Qd[1:]))
        k = np.arange(p, dtype=np.int64)
        Ad = (self.Ad[0] + m, self.Ad[1], self.Ad[2])
        Ac = tuple(cat(t) for t in zip(self.Ac, Ad, (k + m, k + n, -np.ones(p))))
        order = np.lexsort((Ac[1], Ac[0]))
        Ac = tuple(np.ascontiguousarray(a[order]) for a in Ac)
        aug = SparseQCQPFamily(n + p, m + p, 0, self.P, cat([self.q, np.zeros(p)]), self.r, Qc, Ac, cat([self.bc, self.bd]),
                               _EMPTY4, _EMPTY3, np.zeros(0), self.jacobian)
        return aug, cat([x0, self.d_values(x0)]), cat([xl, dl]), cat([xu, du])

    def equalities(self):
        """the same objective and equalities without d(x)"""
        return SparseQCQPFamily(self.n, self.m, 0, self.P, self.q, self.r, self.Qc, self.Ac, self.bc, _EMPTY4, _EMPTY3, np.zeros(0),
                                self.jacobian)

    def d_values(self, x):
        """d(x) = 1/2 x'Qd_k x + Ad_k.x - bd_k (numpy)"""
        x = np.asarray(x, dtype=np.float64)
        mat, r, k, v = self.Qd
        return (0.5 * np.bincount(mat, weights=v * x[r] * x[k], minlength=self.p)
                + _coo_matvec(self.Ad[0], self.Ad[1], self.Ad[2], x, self.p) - self.bd)

    def callbacks(self):
        """numpy callbacks in the conventions of host.optimize_slack: dict(f, grad, hess_vec, c, jac, chess_vec, d, djac,
        dhess_vec).  A reference for tests and the route of a problem through host callbacks; the device path does not use them."""
        n = self.n

        def quad(Qs, Ad, b, cnt):
            mat, r, k, v = Qs

            def val(out, x):
                out[:] = 0.5 * np.bincount(mat, weights=v * x[r] * x[k], minlength=cnt) + _coo_matvec(Ad[0], Ad[1], Ad[2], x, cnt) - b

            def jac(Jc, out, x):
                val(out, x)
                Jc[:, :] = 0.0
                np.add.at(Jc, (mat, r), v * x[k])
                np.add.at(Jc, (Ad[0], Ad[1]), Ad[2])

            def hess(dest, src, x, lam):
                dest[:] = np.bincount(r, weights=lam[mat] * v * src[k], minlength=n)
            return val, jac, hess

        P = self.P

        def f(x):
            return 0.5 * x @ _coo_matvec(P[0], P[1], P[2], x, n) + self.q @ x + self.r

        def grad(g, x):
            g[:] = _coo_matvec(P[0], P[1], P[2], x, n) + self.q

        def hess_vec(dest, src, x):
            dest[:] = _coo_matvec(P[0], P[1], P[2], src, n)

        c, jac, chess = quad(self.Qc, self.Ac, self.bc, self.m)
        d, djac, dhess = quad(self.Qd, self.Ad, self.bd, self.p)
        return dict(f=f, grad=grad, hess_vec=hess_vec, c=c, jac=jac, chess_vec=chess, d=d, djac=djac, dhess_vec=dhess)


_EMPTY3 = (np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0))
_EMPTY4 = (np.zeros(0, np.int64),) + _EMPTY3


def _stack(Ms, name, dims, dn):
    """a sequence of symmetric n x n matrices -> (mat, row, col, val), sorted by (mat, row, col)"""
    parts = []
    for i, M in enumerate(Ms):
        r, k, v, shape = _coo_of(M, "%s[%d]" % (name, i))
        if shape[0] != shape[1]:
            raise _lib.LFPSQPError("sparse_qcqp: %s[%d] must be square, got %s" % (name, i, shape))
        if dims.setdefault("n", shape[0]) != shape[0]:
            raise _lib.LFPSQPError("sparse_qcqp: %s[%d] gives n = %d, another array gives %d" % (name, i, shape[0], dims["n"]))
        r, k, v = _symmetrised(r, k, v, shape[0])
        parts.append((np.full(r.size, i, np.int64), r, k, v))
    if dims.setdefault(dn, len(parts)) != len(parts):
        raise _lib.LFPSQPError("sparse_qcqp: %s has %d matrices, another array gives %s = %d" % (name, len(parts), dn, dims[dn]))
    return tuple(np.concatenate([p[j] for p in parts]) if parts else _EMPTY4[j] for j in range(4))


def sparse_qcqp(P=None, q=None, r=None, Qc=None, Ac=None, bc=None, Qd=None, Ad=None, bd=None, jacobian="dense"):
    """Sparse quadratically constrained quadratic program (large-n mode, one GPU):

        f(x)   = 1/2 x'P x + q.x + r
        c_i(x) = 1/2 x'Qc[i] x + Ac[i].x - bc[i] = 0      i < m
        d_k(x) = 1/2 x'Qd[k] x + Ad[k].x - bd[k] <= 0     k < p   (or dl <= d(x) <= du through optimize_large)

    Matrices are scipy.sparse matrices (anything with .tocoo()) or dense arrays: P (n, n), Ac (m, n), Ad (p, n); Qc and Qd
    are sequences of m and p (n, n) matrices.  None is all zero.  n, m and p are inferred.  Duplicate entries are summed and
    square matrices symmetrised as (M + M')/2, which leaves the quadratic forms unchanged.

    jacobian selects how the device stores the m x n constraint Jacobian.  "dense" (the default) keeps it as a dense array
    (8 m n bytes, twice with bounds); its passes stream all of it and the Gram is a dense DMMA SYRK.  "csr" keeps only its
    structural entries, in CSR and CSC order, and runs the passes and the Gram over that pattern: memory and work scale with
    nnz(J), which lets n grow far beyond what a dense J allows.  Both give the same solution up to rounding.

        fam = families.sparse_qcqp(P=laplacian, Qd=[ball_k ...], bd=radii2 / 2)
        x, obj, lam, info = optimize_large(fam.f, fam.c, fam.d, dl, du, x0, xl, xu, fam.m, fam.p)
    """
    if jacobian not in _JACOBIAN_IDS:
        raise _lib.LFPSQPError('sparse_qcqp: jacobian must be "dense" or "csr", got %r' % (jacobian,))
    dims = {}
    Pc = _EMPTY3
    if P is not None:
        pr, pk, pv, shape = _coo_of(P, "P")
        if shape[0] != shape[1]:
            raise _lib.LFPSQPError("sparse_qcqp: P must be square, got %s" % (shape,))
        dims["n"] = shape[0]
        Pc = _symmetrised(pr, pk, pv, shape[0])
    Qcc = _stack(Qc, "Qc", dims, "m") if Qc is not None else None
    Qdc = _stack(Qd, "Qd", dims, "p") if Qd is not None else None
    lin = {}
    for name, M, dn in (("Ac", Ac, "m"), ("Ad", Ad, "p")):
        if M is None:
            continue
        ar, ak, av, shape = _coo_of(M, name)
        for d, size in ((dn, shape[0]), ("n", shape[1])):
            if dims.setdefault(d, size) != size:
                raise _lib.LFPSQPError("sparse_qcqp: %s gives %s = %d, another array gives %d" % (name, d, size, dims[d]))
        lin[name] = _summed(ar, ak, av, shape[1])
    vecs = {}
    for name, v, dn in (("q", q, "n"), ("bc", bc, "m"), ("bd", bd, "p")):
        if v is None:
            continue
        v = np.asarray(v, dtype=np.float64)
        if v.ndim != 1:
            raise _lib.LFPSQPError("sparse_qcqp: %s must be a vector, got shape %s" % (name, v.shape))
        if dims.setdefault(dn, v.size) != v.size:
            raise _lib.LFPSQPError("sparse_qcqp: %s gives %s = %d, another array gives %d" % (name, dn, v.size, dims[dn]))
        vecs[name] = np.ascontiguousarray(v)
    if "n" not in dims:
        raise _lib.LFPSQPError("sparse_qcqp: n is unknown (give P, q, Qc, Ac, Qd or Ad)")
    n, m, p = dims["n"], dims.get("m", 0), dims.get("p", 0)
    if n < 1:
        raise _lib.LFPSQPError("sparse_qcqp: n must be at least 1")
    if m > 0 and Qc is None and Ac is None:
        raise _lib.LFPSQPError("sparse_qcqp: m = %d equalities need Qc or Ac" % m)
    if p > 0 and Qd is None and Ad is None:
        raise _lib.LFPSQPError("sparse_qcqp: p = %d inequalities need Qd or Ad" % p)
    return SparseQCQPFamily(n, m, p, Pc, vecs.get("q", np.zeros(n)), 0.0 if r is None else float(r),
                            Qcc if Qcc is not None else _EMPTY4, lin.get("Ac", _EMPTY3), vecs.get("bc", np.zeros(m)),
                            Qdc if Qdc is not None else _EMPTY4, lin.get("Ad", _EMPTY3), vecs.get("bd", np.zeros(p)), jacobian)
