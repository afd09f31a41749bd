"""CPU reference for the dense QCQP family: the oracle (oracle/) compiled together with tests/qcqp_reference.cpp, which
adds the family beside the registered ones.  TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The library is compiled on first use, in the oracle's three builds (plain; FMA contraction; left-to-right summation --
the same flags as oracle/Makefile), into a per-user cache directory under the system's temporary directory, so that a
read-only checkout works.  Registered families resolve exactly as in the oracle, inside the same library: comparing an
encoding with its registered family compares two runs of one binary.
"""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

from oracle import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SOURCES = [os.path.join(ROOT, "tests", "qcqp_reference.cpp"), os.path.join(ROOT, "oracle", "lfpsqp_oracle.cpp"),
           os.path.join(ROOT, "oracle", "lfpsqp_oracle.h")]
CXXFLAGS = ["-O3", "-std=c++17", "-fPIC", "-ffp-contract=off", "-w"]
BUILDS = {None: [], "fma": ["-ffp-contract=fast", "-mfma"], "seq": ["-DORC_SEQ_SUM"]}
FAM = dict(O.FAM, qcqp=101)
QCQP_ORDER = ("P", "q", "r", "Qc", "Ac", "bc", "Qd", "Ad", "bd")

_libs = {}
_noise = None


def _paths():
    h = hashlib.sha256()
    for s in SOURCES:
        h.update(open(s, "rb").read())
    h.update(" ".join(CXXFLAGS).encode())
    d = os.path.join(tempfile.gettempdir(), "lfpsqp_qcqp_reference_%d_%s" % (os.getuid(), h.hexdigest()[:16]))
    return d, {b: os.path.join(d, "libqcqp_reference%s.so" % ("" if b is None else "_" + b)) for b in BUILDS}


def build():
    """compile the three builds (in parallel) unless the cache already holds them; returns {build: path}"""
    d, paths = _paths()
    os.makedirs(d, exist_ok=True)
    procs = []
    for b, path in paths.items():
        if os.path.exists(path):
            continue
        tmp = "%s.%d.tmp" % (path, os.getpid())
        cmd = [os.environ.get("CXX", "g++")] + CXXFLAGS + BUILDS[b] + ["-shared", "-o", tmp, SOURCES[0], "-ldl", "-lpthread"]
        procs.append((subprocess.Popen(cmd), tmp, path))
    for p, tmp, path in procs:
        if p.wait() != 0:
            raise RuntimeError("qcqp reference: compiling %s failed" % path)
        os.replace(tmp, path)
    return paths


def lib(build_name=None):
    if build_name not in _libs:
        L = C.CDLL(build()[build_name])
        L.qorc_family_f.restype = C.c_double
        if L.orc_set_lapack(O._find_openblas().encode()) != 0:
            raise RuntimeError("qcqp reference: could not bind dgesvd")
        _libs[build_name] = L
        if _noise is not None:
            L.orc_set_noise(O._dp(_noise), C.c_int64(_noise.shape[1]), C.c_int64(_noise.shape[1] * _noise.shape[2]))
    return _libs[build_name]


def default_params(**kw):
    return O.default_params(**kw)


def set_noise(noise):
    """noise: None, or (B, T, N) rows of randn! for beta > 0 (optimize.jl:264-273), for every build"""
    global _noise
    _noise = None if noise is None else np.ascontiguousarray(noise, dtype=np.float64)
    for L in _libs.values():
        if _noise is None:
            L.orc_set_noise(None, C.c_int64(0), C.c_int64(0))
        else:
            L.orc_set_noise(O._dp(_noise), C.c_int64(_noise.shape[1]), C.c_int64(_noise.shape[1] * _noise.shape[2]))


def qcqp_params(n, m, p, B=None, **arrays):
    """Flat blob [P | q | r | Qc | Ac | bc | Qd | Ad | bd] (zero where an array is absent).  Each array has its own
    shape (shared) or a leading batch axis.  Returns (blob, stride): blob (L,) with stride 0, or (B, L) with stride L."""
    sizes = dict(P=n * n, q=n, r=1, Qc=m * n * n, Ac=m * n, bc=m, Qd=p * n * n, Ad=p * n, bd=p)
    parts = []
    for name in QCQP_ORDER:
        a = arrays.get(name)
        k = sizes[name]
        a = np.zeros(k) if a is None else np.asarray(a, dtype=np.float64)
        parts.append(a.reshape(k) if a.size == k else a.reshape(a.shape[0], k))
    if B is None:
        return np.concatenate(parts), 0
    blob = np.concatenate([np.broadcast_to(a, (B, a.shape[-1])) for a in parts], axis=1)
    return np.ascontiguousarray(blob), blob.shape[1]


def optimize_batched(family, n, m, p, x0, xl=None, xu=None, fam_params=None, fam_stride=0, params=None, H=64,
                     nthreads=1, build=None):
    """as oracle.optimize_batched, with the QCQP family; build = None (plain) | 'fma' | 'seq'"""
    L = lib(build)
    fam = FAM[family] if isinstance(family, str) else family
    prm = params or default_params()
    x0 = O._f64(x0); B = x0.shape[0]
    xl = O._f64(xl); xu = O._f64(xu); fp = O._f64(fam_params)
    x = np.empty((B, n)); obj = np.full((B, H), np.nan); olen = np.zeros(B, dtype=np.int64)
    lam = np.zeros((B, max(m + p, 0))); term = np.zeros(B, dtype=O.TERM_DTYPE); stats = np.zeros(B, dtype=O.STATS_DTYPE)
    rc = L.qorc_optimize_batched(fam, O._dp(fp), C.c_int64(fam_stride), C.c_int64(n), C.c_int64(m), C.c_int64(p),
                                 C.c_int64(B), O._dp(x0), O._dp(xl), O._dp(xu), C.byref(prm), O._dp(x), O._dp(obj),
                                 C.c_int64(H), olen.ctypes.data_as(C.c_void_p), O._dp(lam),
                                 term.ctypes.data_as(C.c_void_p), stats.ctypes.data_as(C.c_void_p), C.c_int(nthreads))
    if rc != 0:
        raise ValueError("qcqp reference optimize_batched failed rc=%d" % rc)
    return x, obj, olen, lam, term, stats


def _fam(family):
    return FAM[family] if isinstance(family, str) else family


def family_f(family, n, m, p, x, fam_params=None, build=None):
    return lib(build).qorc_family_f(_fam(family), O._dp(O._f64(fam_params)), C.c_int64(n), C.c_int64(m), C.c_int64(p),
                                    O._dp(O._f64(x)))


def family_grad(family, n, m, p, x, fam_params=None, build=None):
    g = np.zeros(n)
    lib(build).qorc_family_grad(_fam(family), O._dp(O._f64(fam_params)), C.c_int64(n), C.c_int64(m), C.c_int64(p),
                                O._dp(O._f64(x)), O._dp(g))
    return g


def family_jac(family, n, m, p, x, fam_params=None, build=None):
    J = np.zeros((m + p, n), order="F"); cval = np.zeros(m + p)
    lib(build).qorc_family_jac(_fam(family), O._dp(O._f64(fam_params)), C.c_int64(n), C.c_int64(m), C.c_int64(p),
                               O._dp(O._f64(x)), O._dp(J), O._dp(cval))
    return J, cval


def family_hess(family, n, m, p, x, lam, v, fam_params=None, build=None):
    out = np.zeros(n)
    lib(build).qorc_family_hess(_fam(family), O._dp(O._f64(fam_params)), C.c_int64(n), C.c_int64(m), C.c_int64(p),
                                O._dp(O._f64(x)), O._dp(O._f64(lam)), O._dp(O._f64(v)), O._dp(out))
    return out
