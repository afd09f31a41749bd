"""Batched mode at the edges of its kernel-dispatch tree.

launch_batched_reg (csrc/batched_reg.cu) picks a register-resident instantiation RegSolver<Fam, LW, NPL, ME, INEQ, SPARSE>
from the family, N_A = n + p, the presence of bounds and the lane pattern of the bound kinds; every other shape runs the
shared-memory warp solver (batched_warp.cuh), which switches strategy at ME >= 16, strides several rows per lane once
ME > 32, and is refused by the launcher when one instance does not fit in shared memory.  Every case below states the
kernel it expects (lfpsqp_last_kernel), so that a dispatch change cannot silently move a case to another kernel, and is
judged per instance against three builds of the CPU oracle (tests/parity.py) and against the shared-memory solver.
"""
import ctypes as C
import os

import numpy as np
import pytest

from tests import parity

pytestmark = pytest.mark.gpu

NTHREADS = max(1, min(16, os.cpu_count() or 1))
WARP = (1, 32, 0, 0)


def REG(lw, npl, sparse=0):
    return (2, lw, npl, sparse)


@pytest.fixture(scope="module")
def L():
    import lfpsqp.jl_b200 as L
    L.default_context(0)
    return L


class Case:
    """One batched problem: the device family, the oracle's name for it, inputs and the kernel it must run on."""

    def __init__(self, label, L, name, n, m, p, x0, xl=None, xu=None, params=None, a=None, b=0.0, expect=None, nr=False,
                 maxiter=None):
        self.label, self.name, self.n, self.m, self.p = label, name, n, m, p
        self.x0, self.xl, self.xu, self.expect, self.nr, self.maxiter = x0, xl, xu, expect, nr, maxiter
        self.raw = (params, a, b)
        self.fam = self._family(L, params)

    def _family(self, L, params):
        _, a, b = self.raw
        if self.name == "readme_ineq":
            return L.families.readme_inequality(params)
        if self.name == "readme_eq":
            return L.families.readme_equality(self.n)
        if self.name == "boxquad":
            return L.families.boxquad(params, a=a, b=b)
        if self.name == "sin":
            return L.families.sin_system(self.n, self.m, params)
        if self.name == "thomson":
            return L.families.thomson(self.n // 3)
        if self.name == "diagquad":
            return L.families.diagquad(*params)
        raise ValueError(self.name)

    @property
    def B(self):
        return self.x0.shape[0]

    def prm(self, L):
        kw = dict(do_project_retract=not self.nr)
        if self.maxiter:
            kw["maxiter"] = self.maxiter
        return L.LFPSQPParams(**kw)

    def oprm(self, oracle):
        kw = dict(do_project_retract=0 if self.nr else 1)
        if self.maxiter:
            kw["maxiter"] = self.maxiter
        return oracle.default_params(**kw)

    def args(self, x0, fam=None):
        fam = fam or self.fam
        a = [fam.f, fam.c]
        if self.p:
            a.append(fam.d)
        a.append(x0)
        if self.xl is not None:
            a += [self.xl, self.xu]
        a.append(self.m)
        if self.p:
            a.append(self.p)
        return a

    def gpu(self, L, rows=None, ctx=None):
        """solve (all instances, or the instances `rows`) on the GPU; returns (x, obj, olen, lam, term, stats)"""
        fam, x0 = self.fam, self.x0
        if rows is not None:
            x0 = x0[rows]
            if fam.batched_params:
                fam = self._family(L, self.raw[0][rows])
        return L.optimize_batched(*self.args(x0, fam), self.prm(L), ctx=ctx, return_stats=True)

    def oracle_run(self, oracle, rows=None, x0=None, fam_params=None):
        fp = self.fam.params if fam_params is None else fam_params
        x0 = self.x0 if x0 is None else x0
        if rows is not None:
            x0 = x0[rows]
            if self.fam.batched_params:
                fp = fp[rows]
        stride = fp.shape[1] if (fp is not None and self.fam.batched_params) else 0
        return oracle.optimize_batched(self.name, self.n, self.m, self.p, x0, xl=self.xl, xu=self.xu, fam_params=fp,
                                       fam_stride=stride, params=self.oprm(oracle), nthreads=NTHREADS)

    def oracle_builds(self, oracle):
        out = {"base": self.oracle_run(oracle)}
        for v in ("fma", "seq"):
            with oracle.variant(v):
                out[v] = self.oracle_run(oracle)
        return out

    def probe(self, oracle):
        """the plain oracle on the instances idx with every per-instance input moved by one ulp (up, then down)"""
        def run(idx):
            for to in (np.inf, -np.inf):
                if self.fam.batched_params:
                    yield self.oracle_run(oracle, idx, fam_params=np.nextafter(self.fam.params, to))
                else:
                    yield self.oracle_run(oracle, idx, x0=np.nextafter(self.x0, to))
        return run


def _kernel(L):
    return L.default_context().last_kernel


def _bytes(a):
    return np.ascontiguousarray(a).view(np.uint8)


def _identical(a, b):
    """bitwise equality of every output array (x, obj incl. its NaN tail, obj_len, lambda, term, stats)"""
    for i, (u, v) in enumerate(zip(a, b)):
        if u is None or v is None:
            continue
        if u.shape != v.shape or not np.array_equal(_bytes(u), _bytes(v)):
            return i
    return -1


def _oracle_parity(case, gpu, oracle, extra=None):
    runs = case.oracle_builds(oracle)
    rec = parity.classify(gpu, runs, case.label, probe=case.probe(oracle),
                          extra=dict(kernel=list(case.expect), **(extra or {})))
    parity.record(rec)
    assert rec["status_nonzero"] == 0, parity.fmt_record(rec)
    assert rec["failures"] == 0, (parity.fmt_record(rec), rec["failing_detail"])
    return runs


def _history_err(a, b):
    """per-instance largest difference of the objective histories, relative to the largest |objective| along b's"""
    H = min(a[1].shape[1], b[1].shape[1])
    ao, bo = a[1][:, :H], b[1][:, :H]
    scale = np.nanmax(np.abs(bo), axis=1, keepdims=True) + 1e-300
    return np.nanmax(np.where(np.isnan(bo), 0.0, np.abs(ao - bo)) / scale, axis=1)


# objective values along a truncated run: the iterates before the last are retraction outputs, fixed only to the
# retraction's stopping tolerance; builds of the oracle differ there by up to ~1e-8 of the trajectory's scale (BOXQUAD
# m = 1), so they are held to the x tolerance.  The final objective keeps its 1e-10 bar (parity.classify).
HIST_RTOL = parity.X_RTOL


def _truncated_history(gpu, runs):
    """maxiter-truncated runs: the whole objective history and the termination record follow the reference on every
    instance whose final result does and on which the oracle builds agree (on the others the reference itself is
    rounding-sensitive)"""
    orc = runs["base"]
    stable = parity.within(gpu, orc)
    names = list(runs)
    for i in range(len(names)):
        for j in range(i + 1, len(names)):
            stable &= parity.within(runs[names[j]], runs[names[i]]) & (_history_err(runs[names[j]], runs[names[i]]) <= HIST_RTOL)
    assert stable.mean() >= 0.5, stable.mean()
    g = tuple(a[stable] for a in gpu[:5]); o = tuple(a[stable] for a in orc[:5])
    assert np.all(g[4]["condition"] == o[4]["condition"]) and np.all(g[4]["iter"] == o[4]["iter"])
    assert np.array_equal(g[2], o[2])
    H = min(g[1].shape[1], o[1].shape[1])
    assert np.array_equal(np.isnan(g[1][:, :H]), np.isnan(o[1][:, :H]))
    assert np.max(_history_err(g, o)) <= HIST_RTOL
    for k in ("f_diff", "step_diff"):
        assert np.allclose(g[4][k], o[4][k], rtol=1e-6, atol=1e-12), k


def _vs_smem(L, case, gpu, monkeypatch):
    """the shared-memory solver implements the same reference path: same termination and iteration count, x equal to
    rounding (the bar of test_register_and_shared_memory_kernels_agree)"""
    monkeypatch.setenv("LFPSQP_BATCHED_KERNEL", "smem")
    try:
        sm = case.gpu(L)
        assert _kernel(L) == WARP
    finally:
        monkeypatch.delenv("LFPSQP_BATCHED_KERNEL")
    if case.expect == WARP:   # the variable does not change a problem the warp solver already runs
        assert _identical(gpu, sm) == -1
        return
    same = (gpu[4]["condition"] == sm[4]["condition"]) & (gpu[4]["iter"] == sm[4]["iter"])
    assert same.mean() >= 0.98, same.mean()
    xerr = np.linalg.norm(gpu[0] - sm[0], axis=1) / np.maximum(np.linalg.norm(sm[0], axis=1), 1e-300)
    assert np.max(xerr[same]) < 1e-8, np.max(xerr[same])


# --------------------------------------------------------------------------------------------------------- case table
B_CASE = 64


def _readme_ineq(L, n, expect, seed, xl=None, xu=None, tag="", **kw):
    rng = np.random.default_rng(seed)
    co = rng.standard_normal((B_CASE, n))
    if xl is None:
        xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    return Case("README_INEQ n=%d%s" % (n, tag), L, "readme_ineq", n, 0, 1, np.zeros((B_CASE, n)), xl, xu, params=co,
                expect=expect, **kw)


def _eq_bounds(n, active=True):
    """x_1 in [0.5, 1] keeps c = x_1 - 0.75 feasible; the others cycle none / lower only / upper only / both.  active: the
    one-sided bounds exclude 0, so they hold at the solution; otherwise every bound contains 0 and none is active there"""
    xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    xl[0], xu[0] = 0.5, 1.0
    lo, hi = (0.1, -0.2) if active else (-0.1, 0.2)
    for j in range(1, n):
        k = j % 4
        if k == 1: xl[j] = lo
        elif k == 2: xu[j] = hi
        elif k == 3: xl[j], xu[j] = -0.3, 0.5
    return xl, xu


def _inside(rng, xl, xu, B, margin=0.1):
    """per-instance points strictly inside the box"""
    n = xl.size
    x = rng.standard_normal((B, n))
    lo, hi = np.isfinite(xl), np.isfinite(xu)
    both = lo & hi
    u = rng.uniform(margin, 1 - margin, (B, n))
    fl, fu = np.where(lo, xl, 0.0), np.where(hi, xu, 0.0)
    x = np.where(both, fl + u * (fu - fl), x)
    x = np.where(lo & ~hi, fl + u, x)
    x = np.where(hi & ~lo, fu - u, x)
    return x


def _readme_eq(L, n, bounds, expect, seed, **kw):
    rng = np.random.default_rng(seed)
    if bounds:
        xl, xu = _eq_bounds(n, active=bounds != "interior")
        x0 = _inside(rng, xl, xu, B_CASE)
    else:
        xl = xu = None
        x0 = rng.standard_normal((B_CASE, n))
    tag = (" interior bounds" if bounds == "interior" else " bounds") if bounds else ""
    tag += " NR" if kw.get("nr") else ""
    tag += " maxiter=%d" % kw["maxiter"] if kw.get("maxiter") else ""
    return Case("README_EQ n=%d%s" % (n, tag), L, "readme_eq", n, 1, 0, x0, xl, xu, expect=expect, **kw)


def _box_bounds(n):
    """bound kinds cycle lower only / upper only / both / none, so that slot 1 (variables 16..31) holds every kind"""
    xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    for j in range(n):
        k = j % 4
        if k == 0: xl[j] = -0.5
        elif k == 1: xu[j] = 0.4
        elif k == 2: xl[j], xu[j] = -0.3, 0.6
    return xl, xu


def _boxquad(L, n, m, expect, seed, **kw):
    rng = np.random.default_rng(seed)
    xl, xu = _box_bounds(n)
    # targets inside the box, so that no bound is active at the solution: a bound held at the solution is approached at
    # the rate y -> 0 of the embedding, and where the reference stops along that approach moves beyond 1e-8 under a 1-ulp
    # change of its input on a large share of the instances (no implementation can be judged there)
    t = _inside(rng, xl, xu, B_CASE, margin=0.25)
    x0 = np.tile(np.full(n, 0.25 if m else 0.0), (B_CASE, 1)) + 0.05 * rng.uniform(-1, 1, (B_CASE, n))
    tag = " NR" if kw.get("nr") else ""
    tag += " maxiter=%d" % kw["maxiter"] if kw.get("maxiter") else ""
    return Case("BOXQUAD m=%d n=%d%s" % (m, n, tag), L, "boxquad", n, m, 0, x0, xl, xu, params=t,
                a=np.ones(n) if m else None, b=0.0, expect=expect, **kw)


def _ineq_expect(n):
    NA = n + 1
    if NA <= 32: return REG(16, 2)
    if NA <= 56: return REG(8, 7, 1)
    if NA <= 64: return REG(16, 4)
    if NA <= 128: return REG(32, 4)
    return WARP


SECTION1 = (
    [("ineq", n, {}) for n in (1, 15, 16, 31, 32, 55, 56, 63, 64, 127, 128)]
    + [("ineq", 32, dict(maxiter=3)), ("ineq", 56, dict(maxiter=3)), ("ineq", 64, dict(nr=True)), ("ineq", 16, dict(nr=True))]
    + [("eq", n, dict(bounds=bnd)) for bnd in (False, True) for n in (1, 16, 17, 63, 64, 65)]
    # with bounds held at the solution, NR and truncated runs leave x wherever the reference stops along its approach to the
    # bound: a 1-ulp change of x0 moves the reference's own result beyond 1e-8 on nearly every instance (see _boxquad)
    + [("eq", 63, dict(bounds="interior", nr=True)), ("eq", 17, dict(bounds="interior", maxiter=3)), ("eq", 63, dict(bounds="interior", maxiter=3))]
    + [("box", n, dict(m=m)) for m in (0, 1) for n in (16, 17, 31, 32, 33)]
    + [("box", 31, dict(m=1, nr=True)), ("box", 32, dict(m=0, maxiter=3)), ("box", 17, dict(m=1, maxiter=3))]
)


def _section1_case(L, kind, n, kw, seed):
    kw = dict(kw)
    if kind == "ineq":
        tag = (" NR" if kw.get("nr") else "") + (" maxiter=%d" % kw["maxiter"] if kw.get("maxiter") else "")
        return _readme_ineq(L, n, _ineq_expect(n), seed, tag=tag, **kw)
    if kind == "eq":
        bounds = kw.pop("bounds")
        return _readme_eq(L, n, bounds, REG(16, 4) if n <= 64 else WARP, seed, **kw)
    m = kw.pop("m")
    return _boxquad(L, n, m, REG(16, 2) if n <= 32 else WARP, seed, **kw)


def _id(c):
    kind, n, kw = c
    return "-".join([kind, str(n)] + ["%s=%s" % (k, v) for k, v in sorted(kw.items())])


@pytest.mark.parametrize("spec", SECTION1, ids=[_id(c) for c in SECTION1])
def test_register_kernel_edges_vs_oracle_and_smem(L, oracle, monkeypatch, spec):
    kind, n, kw = spec
    case = _section1_case(L, kind, n, kw, seed=1000 + SECTION1.index(spec))
    gpu = case.gpu(L)
    assert _kernel(L) == case.expect, (case.label, _kernel(L))
    runs = _oracle_parity(case, gpu, oracle)
    if case.maxiter:
        _truncated_history(gpu, runs)
    _vs_smem(L, case, gpu, monkeypatch)


# ------------------------------------------------------------------------- SPARSE / non-SPARSE bound layouts at n = 50
def _c2_layout(bounded):
    """n = 50, N_A = 51: in the LW = 8 layout element j sits in lane j % 8 and the slack (j = 50) in lane 2.  The bounds
    contain the solution -coeff/|coeff| (as in _boxquad, a bound held there makes the reference itself rounding-sensitive)"""
    n = 50
    xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
    for j, kind in bounded:
        if kind == "lower": xl[j] = -0.9
        elif kind == "upper": xu[j] = 0.9
        else: xl[j], xu[j] = -0.9, 0.9
    return xl, xu


LAYOUTS = {
    # parabolas and a circle in the exception slot of lanes 3, 4, 5: still one non-line pair per lane
    "sparse": ([(3, "lower"), (12, "upper"), (21, "both")], REG(8, 7, 1)),
    # a bound on x_10 lands in the slack's lane
    "slack-lane": ([(3, "lower"), (12, "upper"), (21, "both"), (10, "both")], REG(16, 4)),
    # x_3 and x_11 share lane 3
    "two-in-lane": ([(3, "both"), (11, "lower")], REG(16, 4)),
}


@pytest.mark.parametrize("layout", sorted(LAYOUTS))
def test_c2_bound_layouts_vs_oracle_and_smem(L, oracle, monkeypatch, layout):
    bounded, expect = LAYOUTS[layout]
    xl, xu = _c2_layout(bounded)
    case = _readme_ineq(L, 50, expect, seed=77 + sorted(LAYOUTS).index(layout), xl=xl, xu=xu, tag=" bounds " + layout)
    gpu = case.gpu(L)
    assert _kernel(L) == expect, (layout, _kernel(L))
    _oracle_parity(case, gpu, oracle)
    _vs_smem(L, case, gpu, monkeypatch)


# -------------------------------------------------------------------------------- instance independence (bitwise)
def _independence_cases(L):
    rng = np.random.default_rng(5)
    out = [_readme_ineq(L, 20, REG(16, 2), 501), _readme_ineq(L, 50, REG(8, 7, 1), 502),
           _readme_ineq(L, 60, REG(16, 4), 503), _readme_ineq(L, 100, REG(32, 4), 504),
           _readme_eq(L, 40, False, REG(16, 4), 505), _readme_eq(L, 40, True, REG(16, 4), 506),
           _boxquad(L, 20, 0, REG(16, 2), 507), _boxquad(L, 20, 1, REG(16, 2), 508)]
    n, m = 24, 6
    t = rng.standard_normal((B_CASE, n))
    out.append(Case("SIN n=24 m=6", L, "sin", n, m, 0, np.zeros((B_CASE, n)), params=t, expect=WARP))
    return out


INDEP = ["ineq20", "ineq50", "ineq60", "ineq100", "eq40", "eq40-bounds", "box20-m0", "box20-m1", "sin24"]


@pytest.mark.parametrize("which", INDEP)
def test_instances_do_not_depend_on_the_batch(L, which):
    case = _independence_cases(L)[INDEP.index(which)]
    full = case.gpu(L)
    kern = _kernel(L)
    assert kern == case.expect
    groups = 128 // kern[1] if kern[0] == 2 else 8   # instances per CTA (the warp solver runs at most 8 warps per CTA)
    # batches of 1, 2, 3, 5 and one that leaves the last CTA partly filled, at several offsets into the full batch
    for B, off in [(1, 0), (1, 13), (1, case.B - 1), (2, 9), (3, 30), (5, 41), (2 * groups + 3, case.B - 2 * groups - 3)]:
        rows = np.arange(off, off + B)
        sub = case.gpu(L, rows)
        assert _kernel(L) == case.expect
        bad = _identical(sub, tuple(a[rows] for a in full))
        assert bad == -1, (case.label, B, off, ["x", "obj", "obj_len", "lambda", "term", "stats"][bad])
    # shared parameters and the same start: every instance must come out bit-identical
    if case.fam.batched_params:
        shared = Case(case.label + " shared", L, case.name, case.n, case.m, case.p, np.tile(case.x0[3], (2 * groups + 3, 1)),
                      case.xl, case.xu, params=case.raw[0][3], a=case.raw[1], b=case.raw[2], expect=case.expect)
        assert not shared.fam.batched_params
    else:
        shared = Case(case.label + " shared", L, case.name, case.n, case.m, case.p, np.tile(case.x0[3], (2 * groups + 3, 1)),
                      case.xl, case.xu, expect=case.expect)
    res = shared.gpu(L)
    assert _kernel(L) == case.expect
    for r in range(1, shared.B):
        bad = _identical(tuple(a[r:r + 1] for a in res), tuple(a[:1] for a in res))
        assert bad == -1, (shared.label, r, bad)


# ----------------------------------------------------------------------- host pipeline vs device-resident entry point
@pytest.mark.parametrize("B", [16383, 16384, 16385, 65536 + 7])
def test_host_pipeline_matches_device_entry(L, B):
    import torch
    import bench
    from lfpsqp.jl_b200 import _lib
    n, H = bench.N_VARS, bench.HIST
    coeff, x0 = bench.make_inputs(0, B)
    inf = np.inf * np.ones(n)
    ctx = L.default_context()
    fam = L.families.readme_inequality(coeff)
    prm = L.LFPSQPParams().to_c()
    pprm = C.cast(C.pointer(prm), C.c_void_p)
    dev = torch.device("cuda", 0)
    d_coeff = torch.from_numpy(coeff).to(dev); d_x0 = torch.from_numpy(x0).to(dev)

    def device_entry(with_stats):
        d_x = torch.empty((B, n), dtype=torch.float64, device=dev); d_obj = torch.empty((B, H), dtype=torch.float64, device=dev)
        d_len = torch.empty(B, dtype=torch.int64, device=dev); d_lam = torch.empty((B, 1), dtype=torch.float64, device=dev)
        d_term = torch.empty(B * _lib.TERM_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        d_st = torch.empty(B * _lib.STATS_DTYPE.itemsize, dtype=torch.uint8, device=dev) if with_stats else None
        torch.cuda.synchronize()
        ctx.check(ctx.lib.lfpsqp_solve_batched_dev(ctx.h, L.families.README_INEQ, n, 0, 1, B, d_coeff.data_ptr(), n,
                                                   d_x0.data_ptr(), _lib.ptr(-inf), _lib.ptr(inf), pprm, d_x.data_ptr(),
                                                   d_obj.data_ptr(), H, d_len.data_ptr(), d_lam.data_ptr(),
                                                   d_term.data_ptr(), d_st.data_ptr() if with_stats else None))
        out = (d_x.cpu().numpy(), d_obj.cpu().numpy(), d_len.cpu().numpy(), d_lam.cpu().numpy(),
               d_term.cpu().numpy().view(_lib.TERM_DTYPE))
        return out + ((d_st.cpu().numpy().view(_lib.STATS_DTYPE),) if with_stats else (None,))

    def host_entry(with_stats):
        return L.optimize_batched(fam.f, None, fam.d, x0, -inf, inf, 0, 1, history=H, return_stats=with_stats)

    ref = device_entry(True)
    assert _kernel(L) == REG(8, 7, 1)
    olen = np.minimum(ref[2], H)
    assert np.all(np.isnan(ref[1][np.arange(H)[None, :] >= olen[:, None]]))   # the NaN tail past obj_len
    assert _identical(device_entry(False)[:5], ref[:5]) == -1
    runs = {"host": host_entry(True), "host stats=NULL": host_entry(False)}
    for label, out in runs.items():
        assert _kernel(L) == REG(8, 7, 1)
        bad = _identical(tuple(out[:5]) + ((out[5],) if len(out) > 5 else (None,)), ref)
        assert bad == -1, (label, B, ["x", "obj", "obj_len", "lambda", "term", "stats"][bad])


# ------------------------------------------------------------------------------ warp solver beyond one row per lane
def _diagquad_problem(rng, n, m, B, dup=0):
    """shared b; feasible starts: one point moved along the null space of J there (as test_rank_deficient_jacobian_vs_oracle)"""
    Q = rng.standard_normal((m, n)) / np.sqrt(n); A = rng.standard_normal((m, n)) / np.sqrt(n)
    if dup:
        Q[m - dup:] = Q[:dup]; A[m - dup:] = A[:dup]
    xt = rng.standard_normal(n); w = np.exp(rng.uniform(0, np.log(20.0), n))
    x0 = rng.standard_normal(n)
    b = 0.5 * Q @ (x0 * x0) + A @ x0
    J0 = Q * x0[None, :] + A
    P0 = np.eye(n) - np.linalg.pinv(J0) @ J0
    X0 = x0[None, :] + 0.05 * (rng.standard_normal((B, n)) @ P0.T)
    return (Q, A, b, xt, w), X0


DIAG = [(n, m, nr) for n in (33, 97, 200) for m in (15, 16, 33, 40) if m <= n for nr in (False, True)]


@pytest.mark.parametrize("n,m,nr", DIAG)
def test_warp_solver_diagquad_vs_oracle(L, oracle, n, m, nr):
    rng = np.random.default_rng(100 * n + m)
    prm, X0 = _diagquad_problem(rng, n, m, 32)
    case = Case("DIAGQUAD n=%d m=%d%s" % (n, m, " NR" if nr else ""), L, "diagquad", n, m, 0, X0, params=prm,
                expect=WARP, nr=nr)
    gpu = case.gpu(L)
    assert _kernel(L) == WARP
    _oracle_parity(case, gpu, oracle)


@pytest.mark.parametrize("nr", [False, True])
def test_warp_solver_sin_80x40_vs_oracle(L, oracle, nr):
    rng = np.random.default_rng(80)
    n, m, B = 80, 40, 32
    case = Case("SIN n=80 m=40%s" % (" NR" if nr else ""), L, "sin", n, m, 0, np.zeros((B, n)),
                params=rng.standard_normal((B, n)), expect=WARP, nr=nr)
    gpu = case.gpu(L)
    assert _kernel(L) == WARP
    _oracle_parity(case, gpu, oracle)


def test_warp_solver_thomson_20_vs_oracle(L, oracle):
    rng = np.random.default_rng(20)
    B, npts = 32, 20
    x0 = rng.standard_normal((B, npts, 3)); x0 /= np.linalg.norm(x0, axis=2, keepdims=True)
    case = Case("THOMSON 20 points", L, "thomson", 3 * npts, npts, 0, x0.reshape(B, 3 * npts), expect=WARP)
    gpu = case.gpu(L)
    assert _kernel(L) == WARP
    _oracle_parity(case, gpu, oracle)


def test_warp_solver_rank_deficient_40_rows(L, oracle):
    # m = 40 with the last 4 rows copies of the first 4: rank 36 at every iterate, truncated path with ME > 32
    rng = np.random.default_rng(4040)
    n, m, dup = 97, 40, 4
    prm, X0 = _diagquad_problem(rng, n, m, 32, dup=dup)
    case = Case("DIAGQUAD n=97 m=40, 4 duplicated rows", L, "diagquad", n, m, 0, X0, params=prm, expect=WARP)
    gpu = case.gpu(L)
    assert _kernel(L) == WARP
    runs = case.oracle_builds(oracle)
    orc = runs["base"]
    res = parity.compare_batch(gpu, orc, n, case.label)
    print(parity.fmt(res)); print(parity.fmt(parity.compare_batch(runs["fma"], orc, n, case.label + " [oracle+fma vs oracle]")))
    assert np.all(gpu[4]["status"] & 1)
    assert res["cond_frac"] >= 0.95 and res["iter_pm1_frac"] >= 0.9, parity.fmt(res)
    same = gpu[4]["iter"] == orc[4]["iter"]
    xerr = np.linalg.norm(gpu[0] - orc[0], axis=1) / np.linalg.norm(orc[0], axis=1)
    assert same.any() and np.median(xerr[same]) < 1e-7, np.median(xerr[same])
    # minimum-norm multipliers: each pair of copies shares its multiplier equally
    for k in range(dup):
        assert np.allclose(gpu[3][:, k], gpu[3][:, m - dup + k], rtol=1e-6, atol=1e-9), k


def _nomem(L, n, m, nr):
    """B = 1, maxiter = 1 probe of the launcher's shared-memory check: True when the call is refused with ERR_NOMEM"""
    rng = np.random.default_rng(m)
    Q = rng.standard_normal((m, n)) / np.sqrt(n); A = rng.standard_normal((m, n)) / np.sqrt(n)
    fam = L.families.diagquad(Q, A, np.zeros(m), np.zeros(n), np.ones(n))
    try:
        L.optimize_batched(fam.f, fam.c, np.zeros((1, n)), m, L.LFPSQPParams(maxiter=1, do_project_retract=not nr))
    except L.LFPSQPError as e:
        assert "(rc=-6)" in str(e) and "shared memory" in str(e), str(e)
        return True
    return False


@pytest.mark.parametrize("nr", [False, True])
def test_warp_solver_at_the_shared_memory_limit(L, oracle, nr):
    n = 128
    assert not _nomem(L, n, 1, nr) and _nomem(L, n, n, nr)
    lo, hi = 1, n                       # lo fits, hi is refused
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if _nomem(L, n, mid, nr): hi = mid
        else: lo = mid
    m = lo
    print("largest m at n = %d (%s): %d" % (n, "NR" if nr else "PP", m))
    assert m > 32                       # the limit is past one row per lane: the strided paths run at it
    rng = np.random.default_rng(128 + m)
    prm, X0 = _diagquad_problem(rng, n, m, 8)
    case = Case("DIAGQUAD n=128 m=%d (largest that fits, %s)" % (m, "NR" if nr else "PP"), L, "diagquad", n, m, 0, X0,
                params=prm, expect=WARP, nr=nr)
    gpu = case.gpu(L)
    assert _kernel(L) == WARP
    _oracle_parity(case, gpu, oracle, extra=dict(largest_m=m))
    assert _nomem(L, n, m + 1, nr)
    assert _kernel(L)[0] == -1          # nothing was launched
    again = case.gpu(L)                 # the refusal leaves the context usable
    assert _kernel(L) == WARP and _identical(again, gpu) == -1
