"""Batched mode on the dense QCQP family (LFPSQP_FAM_QCQP): every case judged per instance against three builds of the
CPU oracle with the family added (tests/qcqp_reference.py, judged by tests/parity.py), known answers, bit-identity
where the arithmetic is exactly the same, and the argument errors of the C ABI."""
import ctypes as C
import os

import numpy as np
import pytest

from tests import parity
from tests.test_oracle_qcqp import stiefel, sym, trust_region_answer

pytestmark = pytest.mark.gpu

NTHREADS = max(1, min(16, os.cpu_count() or 1))
WARP = (1, 32, 0, 0)
B = 256
# Known answers are checked on runs with a tight KKT and feasibility tolerance.  Parity is judged on the default
# parameters: with eps_f = 0 the stop depends on an objective change of exactly zero, which rounding decides.
TIGHT = dict(eps_kkt=1e-10, eps_f=0.0, eps_c=1e-12, maxiter=2000)


@pytest.fixture(scope="module")
def ref():
    """the CPU oracle with the QCQP family added (tests/qcqp_reference.py), in its three builds"""
    from tests import qcqp_reference
    qcqp_reference.build()
    return qcqp_reference


@pytest.fixture(scope="module")
def L():
    import lfpsqp.jl_b200 as L
    L.default_context(0)
    return L


class Q:
    """One QCQP workload: arrays (own shape = shared, leading axis = per instance), x0 (B, n), optional shared bounds."""

    def __init__(self, label, n, m, p, x0, xl=None, xu=None, **arrays):
        self.label, self.n, self.m, self.p, self.x0 = label, n, m, p, x0
        self.arrays = arrays
        if p and xl is None:
            xl, xu = -np.inf * np.ones(n), np.inf * np.ones(n)
        self.xl, self.xu = xl, xu

    def per_instance(self, name):
        own = {"P": 2, "q": 1, "r": 0, "Qc": 3, "Ac": 2, "bc": 1, "Qd": 3, "Ad": 2, "bd": 1}[name]
        return np.ndim(self.arrays[name]) == own + 1

    def rows(self, rows):
        a = {k: (np.asarray(v)[rows] if self.per_instance(k) else v) for k, v in self.arrays.items()}
        return Q(self.label, self.n, self.m, self.p, self.x0[rows], self.xl, self.xu, **a)

    def fam(self, L):
        return L.families.qcqp(**self.arrays)

    def args(self, fam, x0):
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

    def gpu(self, L, ctx=None, noise=None, **kw):
        return L.optimize_batched(*self.args(self.fam(L), self.x0), L.LFPSQPParams(**kw), ctx=ctx, history=128,
                                  return_stats=True, noise=noise)

    def oracle_run(self, ref, x0=None, build=None, **kw):
        x0 = self.x0 if x0 is None else x0
        sym_arrays = {k: (0.5 * (np.asarray(v) + np.swapaxes(v, -1, -2)) if k in ("P", "Qc", "Qd") else v)
                      for k, v in self.arrays.items()}
        fp, stride = ref.qcqp_params(self.n, self.m, self.p, B=x0.shape[0], **sym_arrays)
        prm = ref.default_params(**{k: int(v) if isinstance(v, bool) else v for k, v in kw.items()})
        return ref.optimize_batched("qcqp", self.n, self.m, self.p, x0, xl=self.xl, xu=self.xu, fam_params=fp,
                                    fam_stride=stride, params=prm, H=128, nthreads=NTHREADS, build=build)

    def judge(self, gpu, ref, label=None, max_fail=0, **kw):
        runs = {"base": self.oracle_run(ref, **kw)}
        for v in ("fma", "seq"):
            runs[v] = self.oracle_run(ref, build=v, **kw)

        def probe(idx):   # the plain oracle with x0 moved by one ulp (up, then down)
            for to in (np.inf, -np.inf):
                yield tuple(a[idx] for a in self.oracle_run(ref, x0=np.nextafter(self.x0, to), **kw)[:5])

        rec = parity.classify(gpu, runs, label or self.label, probe=probe, extra=dict(kernel=list(WARP)))
        parity.record(rec)
        assert rec["failures"] <= max_fail, (parity.fmt_record(rec), rec["failing_detail"])
        return runs


# ------------------------------------------------------------------------------------------------------- workloads
def rayleigh(n=24, seed=1):
    rng = np.random.default_rng(seed)
    A = sym(rng, n)
    x0 = rng.standard_normal((B, n)); x0 /= np.linalg.norm(x0, axis=1, keepdims=True)
    return Q("QCQP Rayleigh n=%d" % n, n, 1, 0, x0, P=A, Qc=2 * np.eye(n)[None], bc=[1.0]), A


def stiefel_case(nrow=8, k=3, seed=2):
    rng = np.random.default_rng(seed)
    A = sym(rng, nrow)
    Qc, bc = stiefel(nrow, k)
    x0 = np.stack([np.linalg.qr(rng.standard_normal((nrow, k)))[0].T.ravel() for _ in range(B)])
    return Q("QCQP Stiefel n=%d m=%d" % (nrow * k, len(bc)), nrow * k, len(bc), 0, x0, P=np.kron(np.eye(k), A), Qc=Qc,
             bc=bc), A


def linear_qp(n=40, m=5, seed=3):
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((B, n, n))
    P = G @ np.swapaxes(G, 1, 2) / n + np.eye(n)
    return Q("QCQP linear-equality QP n=%d m=%d" % (n, m), n, m, 0, rng.standard_normal((B, n)), P=P,
             q=rng.standard_normal(n), Ac=rng.standard_normal((m, n)), bc=rng.standard_normal(m))


def trust_region(n=32, seed=4):
    rng = np.random.default_rng(seed)
    G = rng.standard_normal((B, n, n))
    P = G @ np.swapaxes(G, 1, 2) / n + 0.5 * np.eye(n)
    q = rng.standard_normal((B, n))
    unc = np.linalg.norm(np.linalg.solve(P, q[..., None])[..., 0], axis=1)
    delta = unc * np.where(np.arange(B) % 2 == 0, 2.0, 0.5)     # interior and boundary solutions alternate
    x0 = 0.1 * delta[:, None] * rng.standard_normal((B, n)) / np.sqrt(n)
    return Q("QCQP trust region n=%d" % n, n, 0, 1, x0, P=P, q=q, Qd=np.eye(n)[None], bd=(0.5 * delta ** 2)[:, None]), delta


def mixed(n=30, seed=5):
    """two quadratic equalities (unit sphere, equal norms of the two halves), one quadratic inequality (|x_0| <= 0.2),
    shared box bounds that stay inactive"""
    rng = np.random.default_rng(seed)
    Qc = np.stack([2 * np.eye(n), np.diag(np.r_[np.ones(n // 2), -np.ones(n - n // 2)])])
    Qd = np.zeros((1, n, n)); Qd[0, 0, 0] = 2.0
    x0 = rng.standard_normal((B, n)); x0 /= np.linalg.norm(x0, axis=1, keepdims=True)
    xl, xu = -2.0 * np.ones(n), 2.0 * np.ones(n)
    return Q("QCQP mixed n=%d m=2 p=1 box" % n, n, 2, 1, x0, xl, xu, P=sym(rng, n, spd=True), q=rng.standard_normal(n),
             Qc=Qc, bc=[1.0, 0.0], Qd=Qd, bd=[0.04])


def final_obj(res):
    return res[1][np.arange(res[1].shape[0]), np.minimum(res[2], res[1].shape[1]) - 1]


# ------------------------------------------------------------------------------------------------ parity + answers
def test_rayleigh(L, ref):
    case, A = rayleigh()
    case.judge(case.gpu(L), ref)
    assert L.default_context().last_kernel == WARP
    gpu = case.gpu(L, **TIGHT)
    np.testing.assert_allclose(final_obj(gpu), 0.5 * np.linalg.eigvalsh(A)[0], rtol=1e-9)


def test_stiefel(L, ref):
    case, A = stiefel_case()
    case.judge(case.gpu(L), ref)
    gpu = case.gpu(L, **TIGHT)
    np.testing.assert_allclose(final_obj(gpu), 0.5 * np.linalg.eigvalsh(A)[:3].sum(), rtol=1e-9)


def test_linear_equality_qp_per_instance_P(L, ref):
    case = linear_qp()
    case.judge(case.gpu(L), ref)
    gpu = case.gpu(L, **TIGHT)
    a = case.arrays
    n, m = case.n, case.m
    for k in range(0, B, 37):
        K = np.block([[a["P"][k], a["Ac"].T], [a["Ac"], np.zeros((m, m))]])
        xs = np.linalg.solve(K, np.concatenate([-a["q"], a["bc"]]))[:n]
        assert np.linalg.norm(gpu[0][k] - xs) <= 1e-7 * np.linalg.norm(xs)


def test_trust_region_per_instance(L, ref):
    case, delta = trust_region()
    case.judge(case.gpu(L), ref)
    gpu = case.gpu(L, **TIGHT)
    for k in range(0, B, 17):
        xs = trust_region_answer(case.arrays["P"][k], case.arrays["q"][k], delta[k])
        assert np.linalg.norm(gpu[0][k] - xs) <= 1e-6 * np.linalg.norm(xs)


def test_mixed(L, ref):
    case = mixed()
    gpu = case.gpu(L)
    case.judge(gpu, ref)


def test_rank_deficient_duplicated_constraint(L, ref):
    case, _ = rayleigh(n=24, seed=6)
    case.arrays["Qc"] = np.concatenate([case.arrays["Qc"]] * 2)
    case.arrays["bc"] = [1.0, 1.0]
    case.m = 2
    case.label = "QCQP Rayleigh with a duplicated constraint"
    gpu = case.gpu(L)
    assert np.all(gpu[4]["status"] & 1)       # LFPSQP_ST_RANK_DEFICIENT
    case.judge(gpu, ref)


# ------------------------------------------------------------------------------------------------ driver variants
def _variant_cases():
    return [("rayleigh", lambda: rayleigh()[0]), ("mixed", mixed)]


@pytest.mark.parametrize("which", ["rayleigh", "mixed"])
@pytest.mark.parametrize("variant", ["nr", "exact", "maxiter3"])
def test_driver_variants(L, ref, which, variant):
    case = dict(_variant_cases())[which]()
    kw = dict(nr=dict(do_project_retract=False), exact=dict(linesearch=1), maxiter3=dict(maxiter=3))[variant]
    if which == "mixed" and variant == "nr":
        # with |x_0| <= 0.2 active, NR fails at every step length on some instances, where the reference's armijo! never
        # terminates (linesearch.jl:57-60) and so cannot judge them; NR runs the same problem with the inequality inactive
        case.arrays["bd"] = [2.0]
    gpu = case.gpu(L, **kw)
    # golden-section decisions amplify rounding beyond the x tolerance (as in test_gpu_batched's exact line search
    # test): up to 2 % of the instances may differ from every oracle build there
    runs = case.judge(gpu, ref, label="%s %s" % (case.label, variant), max_fail=B // 50 if variant == "exact" else 0, **kw)
    if variant == "maxiter3":
        orc = runs["base"]
        ok = parity.within(gpu, orc)
        assert ok.mean() >= 0.9
        assert np.array_equal(gpu[4]["condition"][ok], orc[4]["condition"][ok])
        assert np.array_equal(gpu[4]["iter"][ok], orc[4]["iter"][ok])
        assert np.array_equal(gpu[2][ok], orc[2][ok])
        np.testing.assert_allclose(gpu[1][ok, :4], orc[1][ok, :4], rtol=parity.X_RTOL)


@pytest.mark.parametrize("which", ["rayleigh", "mixed"])
def test_beta_noise(L, ref, which):
    case = dict(_variant_cases())[which]()
    N = (2 if case.xl is not None else 1) * (case.n + case.p)
    T = 20
    nz = np.random.default_rng(7).standard_normal((B, T, N))
    kw = dict(beta=1e-3, t_beta=T)
    gpu = case.gpu(L, noise=nz, **kw)
    ref.set_noise(nz)
    try:
        case.judge(gpu, ref, label=case.label + " beta>0", **kw)
    finally:
        ref.set_noise(None)


# ------------------------------------------------------------------------------------------------ bit-identity
def _same(a, b):
    for u, v in zip(a, b):
        if u is None or v is None:
            continue
        assert u.shape == v.shape and np.array_equal(np.ascontiguousarray(u).view(np.uint8),
                                                     np.ascontiguousarray(v).view(np.uint8))


def test_readme_encodings_are_bitwise(L, monkeypatch):
    monkeypatch.setenv("LFPSQP_BATCHED_KERNEL", "smem")
    rng = np.random.default_rng(8)
    n = 50
    x0 = rng.standard_normal((B, n))
    prm = L.LFPSQPParams()
    fam = L.families.readme_equality(n)
    ref = L.optimize_batched(fam.f, fam.c, x0, 1, prm, return_stats=True)
    enc = L.families.qcqp(P=2 * np.eye(n), Ac=np.eye(n)[:1], bc=[0.75])
    _same(L.optimize_batched(enc.f, enc.c, x0, 1, prm, return_stats=True), ref)

    co = rng.standard_normal((B, n)); x0 = 0.1 * rng.standard_normal((B, n)); inf = np.inf * np.ones(n)
    fam = L.families.readme_inequality(co)
    ref = L.optimize_batched(fam.f, None, fam.d, x0, -inf, inf, 0, 1, prm, return_stats=True)
    enc = L.families.qcqp(q=co, Qd=2 * np.eye(n)[None], bd=[1.0])
    _same(L.optimize_batched(enc.f, None, enc.d, x0, -inf, inf, 0, 1, prm, return_stats=True), ref)


def test_diagquad_and_boxquad_encodings(L):
    rng = np.random.default_rng(9)
    n, m = 20, 3
    Qv, A, b = rng.uniform(0.5, 1.5, (m, n)), 0.3 * rng.standard_normal((m, n)), rng.uniform(0.5, 1.0, m)
    xt, w = rng.standard_normal(n), rng.uniform(0.5, 2.0, n)
    x0 = rng.standard_normal((B, n))
    dq = L.families.diagquad(Qv, A, b, xt, w)
    ref = L.optimize_batched(dq.f, dq.c, x0, m)
    enc = L.families.qcqp(P=np.diag(w), q=-w * xt, r=0.5 * np.sum(w * xt ** 2),
                          Qc=np.stack([np.diag(Qv[i]) for i in range(m)]), Ac=A, bc=b)
    got = L.optimize_batched(enc.f, enc.c, x0, m)
    assert parity.within(got, ref).mean() >= 0.98

    t, a = rng.standard_normal(n), rng.standard_normal(n)
    xl, xu = -1.5 * np.ones(n), 1.5 * np.ones(n)
    x0 = rng.uniform(-1, 1, (B, n))
    bq = L.families.boxquad(t, a=a, b=0.2)
    ref = L.optimize_batched(bq.f, bq.c, x0, xl, xu, 1)
    enc = L.families.qcqp(P=2 * np.eye(n), q=-2 * t, r=t @ t, Ac=a[None], bc=[0.2])
    got = L.optimize_batched(enc.f, enc.c, x0, xl, xu, 1)
    assert parity.within(got, ref).mean() >= 0.98


def test_shared_and_replicated_arrays_agree(L):
    case = mixed()
    shared = case.gpu(L)
    rep = {k: np.broadcast_to(v, (B,) + np.shape(v)).copy() for k, v in case.arrays.items()}
    case2 = Q(case.label, case.n, case.m, case.p, case.x0, case.xl, case.xu, **rep)
    _same(case2.gpu(L), shared)


@pytest.mark.parametrize("sizes", [(1, 2, 3, 5), (B - 7,)])
def test_instances_do_not_depend_on_the_batch(L, sizes):
    case = linear_qp(n=40, m=5)
    full = case.gpu(L)
    for nb in sizes:
        rows = np.arange(3, 3 + nb)
        part = case.rows(rows).gpu(L)
        _same(part, tuple(None if a is None else a[rows] for a in full))


@pytest.mark.parametrize("Bn", [300, 16385])
def test_host_and_device_entry_points_agree(L, Bn):
    import torch
    rng = np.random.default_rng(10)
    n, m, p = 12, 1, 1
    P = sym(rng, n, spd=True)[None] + 0.01 * rng.standard_normal((Bn, 1, 1)) * np.eye(n)   # per instance
    arrays = dict(P=P, q=rng.standard_normal(n), Qc=np.eye(n)[None], bc=[1.0], Ad=rng.standard_normal((Bn, 1, n)),
                  bd=[0.3])
    case = Q("host vs dev", n, m, p, rng.standard_normal((Bn, n)), **arrays)
    fam = case.fam(L)
    host = case.gpu(L)
    ctx = L.default_context()
    dev = {k: torch.from_numpy(np.ascontiguousarray(a)).cuda() for k, (a, _) in fam.arrays.items()}
    desc = L._lib.CQcqp()
    for k, (a, per) in fam.arrays.items():
        setattr(desc, k, dev[k].data_ptr()); setattr(desc, k + "_stride", a[0].size if per else 0)
    x0 = torch.from_numpy(case.x0).cuda()
    H = 128
    xo = torch.empty((Bn, n), dtype=torch.float64, device="cuda")
    obj = torch.empty((Bn, H), dtype=torch.float64, device="cuda")
    olen = torch.empty(Bn, dtype=torch.int64, device="cuda")
    lam = torch.empty((Bn, m + p), dtype=torch.float64, device="cuda")
    term = torch.empty((Bn, 40), dtype=torch.uint8, device="cuda")
    stats = torch.empty((Bn, 80), dtype=torch.uint8, device="cuda")
    cp = L.LFPSQPParams().to_c()
    torch.cuda.synchronize()
    xl, xu = case.xl, case.xu
    ctx.check(ctx.lib.lfpsqp_solve_batched_dev(ctx.h, 101, n, m, p, Bn, C.cast(C.pointer(desc), C.c_void_p), 0,
                                               x0.data_ptr(), L._lib.ptr(xl), L._lib.ptr(xu), C.cast(C.pointer(cp), C.c_void_p),
                                               xo.data_ptr(), obj.data_ptr(), H, olen.data_ptr(), lam.data_ptr(),
                                               term.data_ptr(), stats.data_ptr()))
    got = (xo.cpu().numpy(), obj.cpu().numpy(), olen.cpu().numpy(), lam.cpu().numpy(),
           term.cpu().numpy().view(L._lib.TERM_DTYPE)[:, 0], stats.cpu().numpy().view(L._lib.STATS_DTYPE)[:, 0])
    _same(got, host)


def test_multi_gpu_context_matches_one_device(L):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    case, _ = trust_region()
    one = case.gpu(L)
    mctx = L.MultiContext([0, 1])
    _same(case.gpu(L, ctx=mctx), one)


# ------------------------------------------------------------------------------------------------ errors
def _call(L, n, m, p, desc, fam_stride=0, Bn=2, dev=False):
    ctx = L.default_context()
    x0 = np.zeros((Bn, n)); x = np.zeros((Bn, n)); obj = np.zeros((Bn, 8)); olen = np.zeros(Bn, np.int64)
    lam = np.zeros((Bn, m + p)); term = np.zeros(Bn, L._lib.TERM_DTYPE)
    cp = L.LFPSQPParams().to_c()
    fp = None if desc is None else C.cast(C.pointer(desc), C.c_void_p)
    fn = ctx.lib.lfpsqp_solve_batched_dev if dev else ctx.lib.lfpsqp_solve_batched
    return fn(ctx.h, 101, n, m, p, Bn, fp, fam_stride, L._lib.ptr(x0), None, None, C.cast(C.pointer(cp), C.c_void_p),
              L._lib.ptr(x), L._lib.ptr(obj), 8, L._lib.ptr(olen), L._lib.ptr(lam), L._lib.ptr(term), None)


def test_argument_errors(L):
    n = 4
    P = np.eye(n); Pb = np.stack([np.eye(n)] * 2); A = np.ones((1, n))
    ERR_ARG, ERR_FAMILY, ERR_NOMEM = -1, -3, -6

    def desc(**kw):
        d = L._lib.CQcqp()
        for k, (a, s) in kw.items():
            setattr(d, k, a.ctypes.data); setattr(d, k + "_stride", s)
        return d

    assert _call(L, n, 0, 0, None) == ERR_ARG
    assert _call(L, n, 0, 0, desc(P=(P, 0)), fam_stride=3) == ERR_ARG
    assert _call(L, n, 0, 0, desc(P=(Pb, n * n - 1))) == ERR_ARG
    assert _call(L, n, 1, 0, desc(P=(P, 0))) == ERR_ARG                      # m > 0 without Qc / Ac
    assert _call(L, n, 0, 1, desc(P=(P, 0)), dev=True) == ERR_ARG            # p > 0 without Qd / Ad
    Pn = P.copy(); Pn[0, 1] = 0.5
    assert _call(L, n, 0, 0, desc(P=(Pn, 0))) == ERR_ARG                     # not symmetric (host entry point)
    assert _call(L, n, 1, 0, desc(P=(Pb, n * n), Ac=(A, 0))) == 0
    # large-n mode does not take the family
    ctx = L.default_context()
    cp = L.LFPSQPParams().to_c()
    d = desc(P=(P, 0), Ac=(A, 0))
    x = np.zeros(n); obj = np.zeros(8); olen = np.zeros(1, np.int64); lam = np.zeros(1); term = np.zeros(1, L._lib.TERM_DTYPE)
    rc = ctx.lib.lfpsqp_solve_large(ctx.h, 101, n, 1, C.cast(C.pointer(d), C.c_void_p), L._lib.ptr(x), None, None,
                                    C.cast(C.pointer(cp), C.c_void_p), L._lib.ptr(x), L._lib.ptr(obj), 8,
                                    L._lib.ptr(olen), L._lib.ptr(lam), L._lib.ptr(term), None)
    assert rc == ERR_FAMILY
    # one instance beyond the warp solver's shared-memory limit
    nb, mb = 64, 128
    big = desc(Ac=(np.ones((mb, nb)), 0))
    assert _call(L, nb, mb, 0, big) == ERR_NOMEM


def test_python_shape_errors(L):
    with pytest.raises(L.LFPSQPError):
        L.families.qcqp(P=np.eye(3), q=np.ones(4))
    with pytest.raises(L.LFPSQPError):
        L.families.qcqp(P=np.zeros((2, 3, 3)), q=np.zeros((3, 3)))
    with pytest.raises(L.LFPSQPError):
        L.families.qcqp(bc=[1.0])
    with pytest.raises(L.LFPSQPError):
        L.families.qcqp(P=np.eye(3), bc=[1.0])
    fam = L.families.qcqp(P=np.stack([np.eye(3)] * 2))
    with pytest.raises(L.LFPSQPError):
        L.optimize(fam.f, np.ones(3))
